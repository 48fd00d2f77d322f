// The fp32 CUDA-core MLP skeleton of the NeRF and NeuS field variants (SURVEY 8(f) item 3).
//
//   CTA (256 threads) = tile of kT = 64 samples, grid = #SMs, persistent over tiles.  Activations live K-major in
//   shared memory (row = channel, kT columns); a layer reads one or two row segments (e.g. H then E for the layer
//   behind a skip), so concats move no data.  Thread (cg = tid % 16, sg = tid / 16) owns columns 4 sg .. 4 sg + 3
//   and the 16 output channels {4 cg + 64 i + j}: per input row one float4 of activations, four conflict-free float4
//   of weights, 64 FMAs.  Weights: packed once as [in rows, padded to kChunk][256 outputs, padded] fp32, streamed
//   through a double-buffered kChunk-row shared-memory chunk with cp.async; the models stay in L2.
//
// Compiled twice, like the variants' tile programs that include it: by nvcc into the kernels (Ctx = CudaCtx, the CUDA
// thread) and by g++ into tests/emul (Ctx = one of 256 OS threads per CTA, a pthread barrier for __syncthreads), so
// the very same index arithmetic is checked on a machine without a GPU.
#pragma once

#include "common.cuh"

#ifdef __CUDACC__
#define LDG(p) __ldg(p)
#else
#define LDG(p) (*(p))
#endif

namespace neddf {
namespace simt {

constexpr int kT = 64;        // samples per tile
constexpr int kW = 256;       // layer width (fixed)
constexpr int kChunk = 16;    // weight rows per shared-memory chunk
constexpr int kThreads = 256;

struct Layer {
  int w_off;       // float offset of the packed [k_pad][256] block
  int b_off;       // float offset of the [256] bias block
  int k_pad;       // input rows padded to a multiple of kChunk
  int seg_a, n_a;  // first input segment (the variant's enum) and its rows
  int seg_b, n_b;  // second one (0: none)
  int wt_off;      // transposed pack [kt_pad (output channels)][256 (the first 256 input channels)] ...
  int kt_pad;      // ... of a backward pass (0: not packed)
};

// Where a kernel's samples come from: explicit rows pos / dir / var [n, 3] (var may be null), or rays + edges
// (sample n = edge n % n_edges of ray n / n_edges, geometry of Ray.get_sampling_points / get_sampling_cones).
struct Samples {
  int64_t n;
  const float *pos, *dir, *var;
  const float *ray_dir, *ray_orig, *dists;
  int n_edges, sampling_type;
  float ray_radius;
};

// Sample n, or (0, (0, 0, 1), 0) past the end (the padding columns of a ragged tile).
__device__ __forceinline__ void load_sample(const Samples& S, int64_t n, float pos[3], float dir[3], float var[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    pos[i] = 0.f;
    dir[i] = (i == 2) ? 1.f : 0.f;
    var[i] = 0.f;
  }
  if (n >= S.n) return;
  if (S.dists) {
    const int64_t b = n / S.n_edges;
    const int j = (int)(n - b * S.n_edges);
    const float* row = S.dists + b * S.n_edges;
    float o[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      o[i] = S.ray_orig[3 * b + i];
      dir[i] = S.ray_dir[3 * b + i];
    }
    sample_geometry(S.sampling_type, S.ray_radius, o, dir, row[j], far_edge(row, j, S.n_edges), pos, var);
  } else {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      pos[i] = S.pos[3 * n + i];
      dir[i] = S.dir[3 * n + i];
      if (S.var) var[i] = S.var[3 * n + i];
    }
  }
}

// Activation value y and slope d1.  Values as torch's forward computes them (a NaN propagates); slopes as torch
// autograd: relu' = (x > 0), leaky_relu(0.01)' = (x > 0 ? 1 : 0.01); tanhExp: nn_module/tanh_exp.py:26-31 forward,
// :57-60 backward (d = tx - x ex (tx^2 - 1), 1 above the threshold).
__device__ __forceinline__ void act_fd(int act, float x, float& y, float& d1) {
  if (act == NEDDF_ACT_TANHEXP) {
    const float ex = expf(x);
    const float tx = tanhf(ex);
    y = x * tx;
    d1 = tx - x * ex * (tx * tx - 1.0f);
    if (x > 20.0f) {
      y = x;
      d1 = 1.0f;
    }
  } else if (act == NEDDF_ACT_RELU) {
    y = x * ((x >= 0.0f) ? 1.0f : 0.0f);
    d1 = (x > 0.0f) ? 1.0f : 0.0f;
  } else {
    y = x * ((x < 0.0f) ? 0.01f : 1.0f);
    d1 = (x > 0.0f) ? 1.0f : 0.01f;
  }
}

// acc[i][j][col] = sum_k W[k][4 cg + 64 i + j] * in[k][4 sg + col], where input row k < n_a is row k of A and the
// next n_b rows are those of B; wl = the packed [k_pad][256] block, Wc = the [2][kChunk][kW] chunk buffers.
// Entry: every thread has passed a barrier after the last write to A / B and after the last read of Wc.
// Exit: every thread has finished reading A / B (trailing barrier).
template <class Ctx>
__device__ __forceinline__ void layer_gemm(Ctx& cx, const float* wl, int k_pad, const float* A, int n_a, const float* B, int n_b,
                                           float* Wc, float (&acc)[4][4][4]) {
  const int tid = cx.tid;
  const int cg = tid & 15, sg = tid >> 4;
  const int n_chunks = k_pad / kChunk;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int s = 0; s < 4; ++s) acc[i][j][s] = 0.f;
  auto load_chunk = [&](int buf, int c) {
    const float* src = wl + (size_t)c * kChunk * kW;
    float* dst = Wc + buf * kChunk * kW;
#pragma unroll
    for (int u = 0; u < (kChunk * kW / 4) / kThreads; ++u) cx.cp16(dst + 4 * (tid + u * kThreads), src + 4 * (tid + u * kThreads));
    cx.cp_commit();
  };
  load_chunk(0, 0);
  for (int c = 0; c < n_chunks; ++c) {
    if (c + 1 < n_chunks) {
      load_chunk((c + 1) & 1, c + 1);
      cx.cp_wait_1();
    } else {
      cx.cp_wait_0();
    }
    cx.sync();
    const float* wc = Wc + (c & 1) * kChunk * kW;
#pragma unroll 4
    for (int kk = 0; kk < kChunk; ++kk) {
      const int k = c * kChunk + kk;
      // rows beyond the layer's inputs carry zero weights; they read row 0 of the first segment
      const float* rowp = (k < n_a) ? A + k * kT : ((k < n_a + n_b) ? B + (k - n_a) * kT : A);
      const float4 a = *reinterpret_cast<const float4*>(rowp + 4 * sg);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 w4 = *reinterpret_cast<const float4*>(wc + kk * kW + 4 * cg + 64 * i);
        const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j][0] = fmaf(wv[j], a.x, acc[i][j][0]);
          acc[i][j][1] = fmaf(wv[j], a.y, acc[i][j][1]);
          acc[i][j][2] = fmaf(wv[j], a.z, acc[i][j][2]);
          acc[i][j][3] = fmaf(wv[j], a.w, acc[i][j][3]);
        }
      }
    }
    cx.sync();  // chunk buffer free; after the last chunk: every thread is done reading A / B
  }
}

// torch Linear weight w [n_out][n_in] -> entry (k, c) of the forward pack [k_pad][256] ...
__device__ __forceinline__ float pack_fwd(const float* w, int n_in, int n_out, int k, int c) {
  return (k < n_in && c < n_out) ? w[(size_t)c * n_in + k] : 0.f;
}
// ... and of the transposed pack [kt_pad][256]: the first 256 input channels (the h part) of output row k
__device__ __forceinline__ float pack_bwd(const float* w, int n_in, int n_out, int k, int c) {
  return (k < n_out && c < n_in && c < kW) ? w[(size_t)k * n_in + c] : 0.f;
}

// config->skips names layer `lid` (the concat [h | E] follows it)
template <class Config>
inline bool is_skip(const Config* c, int lid) {
  for (int i = 0; i < c->n_skips; ++i)
    if (c->skips[i] == lid) return true;
  return false;
}

#ifdef __CUDACC__
struct CudaCtx {
  int tid, block, nblocks;
  __device__ __forceinline__ void sync() { __syncthreads(); }
  __device__ __forceinline__ void cp16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
  }
  __device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
  __device__ __forceinline__ void cp_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
  __device__ __forceinline__ void cp_wait_0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
};

// One torch nn.Linear (w [n_out][n_in], b [n_out]) into its blocks of the packed buffer dst: the forward pack, the bias
// and, when ly.kt_pad > 0, the transposed pack.
static __global__ void pack_layer_kernel(const float* __restrict__ w, const float* __restrict__ b, int n_in, int n_out, Layer ly,
                                         float* __restrict__ dst) {
  const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int idx = t0; idx < ly.k_pad * kW; idx += stride) dst[ly.w_off + idx] = pack_fwd(w, n_in, n_out, idx / kW, idx % kW);
  for (int idx = t0; idx < ly.kt_pad * kW; idx += stride) dst[ly.wt_off + idx] = pack_bwd(w, n_in, n_out, idx / kW, idx % kW);
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < kW; c += blockDim.x) dst[ly.b_off + c] = c < n_out ? b[c] : 0.f;
}
#endif

}  // namespace simt
}  // namespace neddf
