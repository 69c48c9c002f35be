// Spectral normalisation of the decoder layers (torch.nn.utils.spectral_norm with dim=0, one power
// iteration, eps=1e-12; model.py:334-344 with sn: True): the power iteration + W/sigma in front of the
// existing conv / linear kernels, and the sigma correction of their weight gradient behind them.
//
// One CTA per layer: within a layer the chain W^T u -> norm -> W v -> norm -> dot is serial, and the
// largest decoder layer is only 256 x 640 floats.  A single CTA is bound by the loads it keeps in flight,
// so every pass reads float4s (when the layer's rows are 16-byte aligned) with several independent
// accumulators per thread.  Every reduction still runs in a fixed order (fixed per-thread partials,
// xor-shuffle warp sums, per-warp partials summed by one thread), never through atomics, so u, v, sigma
// and the outputs are bit-identical from run to run -- and across data-parallel replicas, which must
// stay identical.
#include "common.cuh"

namespace avc {

constexpr int SN_THREADS = 512;
constexpr int SN_WARPS = SN_THREADS / 32;
constexpr int SN_UNROLL = 4;
constexpr float SN_EPS = 1e-12f;

// Sum of `v` over the CTA in a fixed order; every thread receives the total.  `red` holds SN_WARPS + 1 floats.
__device__ float sn_block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();   // `red` may still be read by the previous call
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < SN_WARPS; ++w) s += red[w];
    red[SN_WARPS] = s;
  }
  __syncthreads();
  return red[SN_WARPS];
}

template <int V>
__device__ __forceinline__ void ldv(const float* p, float* o) {
  if constexpr (V == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  } else {
    o[0] = *p;
  }
}

// s[i] = sum_j W[i][j] x[j] for every row (one warp per row, each lane V columns per step and SN_UNROLL steps in
// flight), stored to out[i] unless out is null; returns, to every thread, sum_i s[i] * y[i] (y = s when y is null).
template <int V>
__device__ float sn_rows(const float* __restrict__ W, int rows, int cols, const float* x, float* out, const float* y,
                         float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int STEP = 32 * V;
  float part = 0.f;
  for (int i = warp; i < rows; i += SN_WARPS) {
    const float* wr = W + (int64_t)i * cols;
    float acc[SN_UNROLL] = {};
    int j = lane * V;
    for (; j + (SN_UNROLL - 1) * STEP < cols; j += SN_UNROLL * STEP) {
      float w[SN_UNROLL][V], xv[SN_UNROLL][V];
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q) {
        ldv<V>(wr + j + q * STEP, w[q]);
        ldv<V>(x + j + q * STEP, xv[q]);
      }
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q)
#pragma unroll
        for (int e = 0; e < V; ++e) acc[q] += w[q][e] * xv[q][e];
    }
    for (; j < cols; j += STEP) {
      float w[V], xv[V];
      ldv<V>(wr + j, w);
      ldv<V>(x + j, xv);
#pragma unroll
      for (int e = 0; e < V; ++e) acc[0] += w[e] * xv[e];
    }
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < SN_UNROLL; ++q) s += acc[q];
    s = warp_sum(s);
    if (lane == 0 && out) out[i] = s;
    part += s * (y ? y[i] : s);
  }
  // lanes hold identical `part`: count lane 0's only
  return sn_block_sum(lane == 0 ? part : 0.f, red);
}

// out[j] = sum_i W[i][j] x[i] for every column: a lane covers V columns (a warp 32 * V), the warps split the rows
// (SN_UNROLL rows in flight per thread), and the SN_WARPS partials of a column are summed in warp order.  Returns
// sum_j out[j]^2 to every thread.  `part` holds SN_WARPS * 32 * V floats.
template <int V>
__device__ float sn_cols(const float* __restrict__ W, int rows, int cols, const float* x, float* out, float* part,
                         float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int STEP = SN_WARPS;
  float sq = 0.f;
  for (int j0 = 0; j0 < cols; j0 += 32 * V) {
    const int j = j0 + lane * V;
    float acc[SN_UNROLL][V] = {};
    if (j < cols) {
      int i = warp;
      for (; i + (SN_UNROLL - 1) * STEP < rows; i += SN_UNROLL * STEP) {
        float w[SN_UNROLL][V], xi[SN_UNROLL];
#pragma unroll
        for (int q = 0; q < SN_UNROLL; ++q) {
          ldv<V>(W + (int64_t)(i + q * STEP) * cols + j, w[q]);
          xi[q] = x[i + q * STEP];
        }
#pragma unroll
        for (int q = 0; q < SN_UNROLL; ++q)
#pragma unroll
          for (int e = 0; e < V; ++e) acc[q][e] += w[q][e] * xi[q];
      }
      for (; i < rows; i += STEP) {
        float w[V];
        ldv<V>(W + (int64_t)i * cols + j, w);
        const float xi = x[i];
#pragma unroll
        for (int e = 0; e < V; ++e) acc[0][e] += w[e] * xi;
      }
    }
#pragma unroll
    for (int e = 0; e < V; ++e) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q) s += acc[q][e];
      part[warp * 32 * V + lane * V + e] = s;
    }
    __syncthreads();
    if (warp == 0 && j < cols) {
#pragma unroll
      for (int e = 0; e < V; ++e) {
        float t = 0.f;
        for (int w = 0; w < SN_WARPS; ++w) t += part[w * 32 * V + lane * V + e];
        out[j + e] = t;
        sq += t * t;
      }
    }
    __syncthreads();
  }
  return sn_block_sum(sq, red);
}

__device__ __forceinline__ bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

template <int V>
__device__ void sn_fwd_layer(const avc_sn_item& it, int update, float* part, float* red) {
  const int rows = it.rows, cols = it.cols;
  const float* W = it.w_orig;
  float* u = it.u;
  float* v = it.v;
  // u and v are written and re-read by this CTA only: __syncthreads orders those global accesses
  float sigma;
  if (update) {
    // v = normalize(W^T u)
    const float inv_v = 1.f / fmaxf(sqrtf(sn_cols<V>(W, rows, cols, u, v, part, red)), SN_EPS);
    for (int j = threadIdx.x; j < cols; j += SN_THREADS) v[j] *= inv_v;
    __syncthreads();
    // s = W v; u = normalize(s); sigma = u . s
    const float ss = sn_rows<V>(W, rows, cols, v, u, nullptr, red);
    const float inv_u = 1.f / fmaxf(sqrtf(ss), SN_EPS);
    for (int i = threadIdx.x; i < rows; i += SN_THREADS) u[i] *= inv_u;
    sigma = ss * inv_u;
  } else {
    // sigma = u . (W v) from the stored vectors
    sigma = sn_rows<V>(W, rows, cols, v, nullptr, u, red);
  }
  if (threadIdx.x == 0) *it.sigma = sigma;
  const int64_t n = (int64_t)rows * cols;
  if constexpr (V == 4) {
    const float4* w4 = reinterpret_cast<const float4*>(W);
    float4* o4 = reinterpret_cast<float4*>(it.w_sn);
    const int64_t n4 = n / 4;
    int64_t k = threadIdx.x;
    for (; k + (SN_UNROLL - 1) * SN_THREADS < n4; k += SN_UNROLL * SN_THREADS) {
      float4 t[SN_UNROLL];
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q) t[q] = w4[k + q * SN_THREADS];
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q)
        o4[k + q * SN_THREADS] = make_float4(t[q].x / sigma, t[q].y / sigma, t[q].z / sigma, t[q].w / sigma);
    }
    for (; k < n4; k += SN_THREADS) {
      const float4 t = w4[k];
      o4[k] = make_float4(t.x / sigma, t.y / sigma, t.z / sigma, t.w / sigma);
    }
  } else {
    for (int64_t k = threadIdx.x; k < n; k += SN_THREADS) it.w_sn[k] = W[k] / sigma;
  }
}

__global__ void __launch_bounds__(SN_THREADS) spectral_norm_fwd_kernel(const avc_sn_item* __restrict__ items, int update) {
  __shared__ float part[SN_WARPS * 32 * 4];
  __shared__ float red[SN_WARPS + 1];
  const avc_sn_item it = items[blockIdx.x];
  if (it.rows <= 0 || it.cols <= 0) return;
  if (it.cols % 4 == 0 && aligned16(it.w_orig) && aligned16(it.w_sn) && aligned16(it.v))
    sn_fwd_layer<4>(it, update, part, red);
  else
    sn_fwd_layer<1>(it, update, part, red);
}

__global__ void __launch_bounds__(SN_THREADS) spectral_norm_bwd_kernel(const avc_sn_item* __restrict__ items) {
  __shared__ float red[SN_WARPS + 1];
  const avc_sn_item it = items[blockIdx.x];
  const int rows = it.rows, cols = it.cols;
  if (rows <= 0 || cols <= 0) return;
  const int64_t n = (int64_t)rows * cols;
  float* g = it.grad;
  const float* wsn = it.w_sn;
  const float* u = it.u;
  const float* v = it.v;
  const bool vec = cols % 4 == 0 && aligned16(g) && aligned16(wsn);
  // <grad, w_sn>: SN_UNROLL independent partials per thread, added in a fixed order
  float acc[SN_UNROLL] = {};
  if (vec) {
    const float4* g4 = reinterpret_cast<const float4*>(g);
    const float4* w4 = reinterpret_cast<const float4*>(wsn);
    const int64_t n4 = n / 4;
    int64_t k = threadIdx.x;
    for (; k + (SN_UNROLL - 1) * SN_THREADS < n4; k += SN_UNROLL * SN_THREADS) {
      float4 a[SN_UNROLL], b[SN_UNROLL];
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q) {
        a[q] = g4[k + q * SN_THREADS];
        b[q] = w4[k + q * SN_THREADS];
      }
#pragma unroll
      for (int q = 0; q < SN_UNROLL; ++q) acc[q] += a[q].x * b[q].x + a[q].y * b[q].y + a[q].z * b[q].z + a[q].w * b[q].w;
    }
    for (; k < n4; k += SN_THREADS) {
      const float4 a = g4[k], b = w4[k];
      acc[0] += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
    }
  } else {
    for (int64_t k = threadIdx.x; k < n; k += SN_THREADS) acc[0] += g[k] * wsn[k];
  }
  float dot = 0.f;
#pragma unroll
  for (int q = 0; q < SN_UNROLL; ++q) dot += acc[q];
  dot = sn_block_sum(dot, red);
  const float inv = 1.f / *it.sigma;
  // grad = (grad - <grad, w_sn> u v^T) / sigma
  if (vec) {
    float4* g4 = reinterpret_cast<float4*>(g);
    const int64_t n4 = n / 4;
    for (int64_t k = threadIdx.x; k < n4; k += SN_THREADS) {
      const int64_t e0 = 4 * k;
      const int i = (int)(e0 / cols), j = (int)(e0 - (int64_t)i * cols);   // cols % 4 == 0: one row
      const float du = dot * u[i];
      float4 t = g4[k];
      t.x = (t.x - du * v[j]) * inv;
      t.y = (t.y - du * v[j + 1]) * inv;
      t.z = (t.z - du * v[j + 2]) * inv;
      t.w = (t.w - du * v[j + 3]) * inv;
      g4[k] = t;
    }
  } else {
    for (int64_t k = threadIdx.x; k < n; k += SN_THREADS) {
      const int i = (int)(k / cols), j = (int)(k - (int64_t)i * cols);
      g[k] = (g[k] - dot * u[i] * v[j]) * inv;
    }
  }
}

}  // namespace avc

using namespace avc;

extern "C" int avc_spectral_norm_fwd(const avc_sn_item* items_dev, int n_items, int update, void* stream) {
  AVC_REQUIRE(items_dev && n_items > 0, AVC_ERR_INVALID, "avc_spectral_norm_fwd: bad argument");
  AVC_LAUNCH(spectral_norm_fwd_kernel, n_items, SN_THREADS, 0, (cudaStream_t)stream, items_dev, update ? 1 : 0);
  AVC_CHECK_LAUNCH("spectral_norm_fwd");
  return AVC_OK;
}

extern "C" int avc_spectral_norm_bwd(const avc_sn_item* items_dev, int n_items, void* stream) {
  AVC_REQUIRE(items_dev && n_items > 0, AVC_ERR_INVALID, "avc_spectral_norm_bwd: bad argument");
  AVC_LAUNCH(spectral_norm_bwd_kernel, n_items, SN_THREADS, 0, (cudaStream_t)stream, items_dev);
  AVC_CHECK_LAUNCH("spectral_norm_bwd");
  return AVC_OK;
}
