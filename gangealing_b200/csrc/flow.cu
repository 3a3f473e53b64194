// flow.cu -- flow composition of the flow STN head in one pass, forward and backward (sm_100a).
//
// Replaces ~20 ATen launches of reference models/spatial_transformers/warping_heads.py:
//   upsample_flow (:180-193)  softmax over the 9 mask logits, F.unfold(8*flow, 3x3), weighted sum, 2 permutes
//   FlowHead.forward (:239-244) flow = identity_flow + delta_flow; apply_affine(base_warp, flow) (:268-277);
//                               identity_flow.lerp(flow, alpha)
// One thread per full-resolution flow pixel; tensors are KB-sized, so the cost is launch latency and the
// win is launch count.  Algorithmic bytes per sample (K=1, 16x16 -> 128x128): mask 0.59 MB + outputs 0.26 MB.
#include "common.cuh"

namespace gg {
namespace {

struct FlowParams {
  int64_t n;       // samples (N*K)
  int h, w;        // low-res size
  int s;           // flow_downsample (8)
};

// index helpers: mask is (N, 9*s*s, H, W) viewed (N, 9, s, s, H, W) (warping_heads.py:184)
__device__ __forceinline__ int64_t mask_index(const FlowParams& p, int64_t n, int k, int sy, int sx, int h, int w) {
  return ((((n * 9 + k) * p.s + sy) * p.s + sx) * p.h + h) * static_cast<int64_t>(p.w) + w;
}

// thread index -> (n, sy, sx, h, w) in mask memory order (w fastest): coalesced mask reads
__device__ __forceinline__ void decode(const FlowParams& p, int64_t idx, int64_t& n, int& sy, int& sx, int& h, int& w) {
  w = static_cast<int>(idx % p.w); idx /= p.w;
  h = static_cast<int>(idx % p.h); idx /= p.h;
  sx = static_cast<int>(idx % p.s); idx /= p.s;
  sy = static_cast<int>(idx % p.s); idx /= p.s;
  n = idx;
}

__global__ void __launch_bounds__(256)
flow_compose_fwd_kernel(float* __restrict__ delta_out, float* __restrict__ flow_out, const float* __restrict__ low,
                        const float* __restrict__ mask, const float* __restrict__ identity,
                        const float* __restrict__ base, const float* __restrict__ alpha, FlowParams p, int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t n; int sy, sx, h, w;
    decode(p, idx, n, sy, sx, h, w);
    // softmax over the 9 logits
    float lg[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) { lg[k] = mask[mask_index(p, n, k, sy, sx, h, w)]; mx = fmaxf(mx, lg[k]); }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { lg[k] = expf(lg[k] - mx); sum += lg[k]; }
    const float inv = 1.f / sum;
    // convex combination of the 3x3 neighbourhood of s*flow (zero padded, F.unfold padding=1)
    float dx = 0.f, dy = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int hh = h + k / 3 - 1, ww = w + k % 3 - 1;
      if (hh >= 0 && hh < p.h && ww >= 0 && ww < p.w) {
        const float2 f = *reinterpret_cast<const float2*>(low + ((n * p.h + hh) * static_cast<int64_t>(p.w) + ww) * 2);
        const float pk = lg[k] * inv;
        dx = fmaf(pk, static_cast<float>(p.s) * f.x, dx);
        dy = fmaf(pk, static_cast<float>(p.s) * f.y, dy);
      }
    }
    const int Y = h * p.s + sy, X = w * p.s + sx;
    const int64_t pix = (static_cast<int64_t>(Y) * (p.w * p.s) + X) * 2;
    const int64_t o = n * (p.h * p.s) * static_cast<int64_t>(p.w * p.s) * 2 + pix;
    *reinterpret_cast<float2*>(delta_out + o) = make_float2(dx, dy);
    if (flow_out) {
      const float2 id = *reinterpret_cast<const float2*>(identity + pix);
      float gx = id.x + dx, gy = id.y + dy;
      if (base) {  // [gx, gy, 1] @ M^T   (warping_heads.py:268-277)
        const float* M = base + n * 6;
        const float tx = M[0] * gx + M[1] * gy + M[2];
        const float ty = M[3] * gx + M[4] * gy + M[5];
        gx = tx; gy = ty;
      }
      if (alpha) {  // identity.lerp(flow, alpha) = identity + alpha*(flow - identity)
        const float a = alpha[n];
        gx = id.x + a * (gx - id.x);
        gy = id.y + a * (gy - id.y);
      }
      *reinterpret_cast<float2*>(flow_out + o) = make_float2(gx, gy);
    }
  }
}

// backward: g_delta (direct, may be null) and g_flow (may be null) -> g_mask (written); the per-pixel terms of g_low
// (one per tap) and of g_base (6 per pixel) go to the caller's workspace, and flow_low_gather_kernel /
// flow_base_reduce_kernel sum them in a fixed order (no float atomics: the same bits on every run).  The g_low terms are
// laid out by the low-res cell they belong to, (N, H, W, 9, S, S): each cell's terms are contiguous.
__global__ void __launch_bounds__(256)
flow_compose_bwd_kernel(float* __restrict__ g_mask, float2* __restrict__ g_low, float* __restrict__ g_base,
                        const float* __restrict__ g_delta, const float* __restrict__ g_flow,
                        const float* __restrict__ low, const float* __restrict__ mask,
                        const float* __restrict__ identity, const float* __restrict__ base,
                        const float* __restrict__ alpha, FlowParams p, int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t n; int sy, sx, h, w;
    decode(p, idx, n, sy, sx, h, w);
    const int Y = h * p.s + sy, X = w * p.s + sx;
    const int64_t pix = (static_cast<int64_t>(Y) * (p.w * p.s) + X) * 2;
    const int64_t o = n * (p.h * p.s) * static_cast<int64_t>(p.w * p.s) * 2 + pix;
    // recompute softmax and the neighbourhood
    float pk[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) { pk[k] = mask[mask_index(p, n, k, sy, sx, h, w)]; mx = fmaxf(mx, pk[k]); }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { pk[k] = expf(pk[k] - mx); sum += pk[k]; }
    const float inv = 1.f / sum;
    float fx[9], fy[9];
    float dx = 0.f, dy = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      pk[k] *= inv;
      const int hh = h + k / 3 - 1, ww = w + k % 3 - 1;
      fx[k] = 0.f; fy[k] = 0.f;
      if (hh >= 0 && hh < p.h && ww >= 0 && ww < p.w) {
        const float2 f = *reinterpret_cast<const float2*>(low + ((n * p.h + hh) * static_cast<int64_t>(p.w) + ww) * 2);
        fx[k] = static_cast<float>(p.s) * f.x; fy[k] = static_cast<float>(p.s) * f.y;
      }
      dx = fmaf(pk[k], fx[k], dx); dy = fmaf(pk[k], fy[k], dy);
    }
    // gradient arriving at delta
    float gdx = 0.f, gdy = 0.f;
    if (g_delta) { const float2 g = *reinterpret_cast<const float2*>(g_delta + o); gdx = g.x; gdy = g.y; }
    if (g_flow) {
      float2 gf = *reinterpret_cast<const float2*>(g_flow + o);
      if (alpha) { const float a = alpha[n]; gf.x *= a; gf.y *= a; }
      if (base) {
        const float2 id = *reinterpret_cast<const float2*>(identity + pix);
        const float gx = id.x + dx, gy = id.y + dy;
        const float* M = base + n * 6;
        if (g_base) {
          float* gb = g_base + idx * 6;
          gb[0] = gf.x * gx; gb[1] = gf.x * gy; gb[2] = gf.x;
          gb[3] = gf.y * gx; gb[4] = gf.y * gy; gb[5] = gf.y;
        }
        const float px = M[0] * gf.x + M[3] * gf.y;
        const float py = M[1] * gf.x + M[4] * gf.y;
        gf.x = px; gf.y = py;
      }
      gdx += gf.x; gdy += gf.y;
    }
    // through the convex combination: d/dlogit_k = p_k (t_k - sum_j p_j t_j), t_k = <g, f_k>
    float t[9], tbar = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { t[k] = gdx * fx[k] + gdy * fy[k]; tbar = fmaf(pk[k], t[k], tbar); }
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      if (g_mask) g_mask[mask_index(p, n, k, sy, sx, h, w)] = pk[k] * (t[k] - tbar);
      if (g_low) {
        const int hh = h + k / 3 - 1, ww = w + k % 3 - 1;
        if (hh >= 0 && hh < p.h && ww >= 0 && ww < p.w) {
          const float sc = static_cast<float>(p.s) * pk[k];
          const int64_t cell = (n * p.h + hh) * static_cast<int64_t>(p.w) + ww;
          g_low[((cell * 9 + k) * p.s + sy) * p.s + sx] = make_float2(sc * gdx, sc * gdy);
        }
      }
    }
  }
}

// g_low[n, hh, ww] = sum of the 9*S*S terms of low-res cell (hh, ww) (taps whose source cell is outside the grid have
// none): one warp per cell, coalesced reads, lane-strided sums and a shuffle tree -- a fixed order
__global__ void __launch_bounds__(256)
flow_low_gather_kernel(float* __restrict__ g_low, const float2* __restrict__ terms, FlowParams p, int64_t cells) {
  const int lane = threadIdx.x & 31;
  const int ss = p.s * p.s;
  for (int64_t c = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; c < cells;
       c += (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5) {
    const int ww = static_cast<int>(c % p.w);
    const int hh = static_cast<int>((c / p.w) % p.h);
    const float2* t = terms + c * 9 * ss;
    float gx = 0.f, gy = 0.f;
    for (int e = lane; e < 9 * ss; e += 32) {
      const int k = e / ss;
      const int h = hh - (k / 3 - 1), w = ww - (k % 3 - 1);
      if (h < 0 || h >= p.h || w < 0 || w >= p.w) continue;
      const float2 v = t[e];
      gx += v.x; gy += v.y;
    }
    gx = warp_sum(gx);
    gy = warp_sum(gy);
    if (lane == 0) *reinterpret_cast<float2*>(g_low + c * 2) = make_float2(gx, gy);
  }
}

// g_base[n, q] = sum of the 6 per-pixel terms over sample n: one block per sample, fixed-order tree reduction
__global__ void __launch_bounds__(256)
flow_base_reduce_kernel(float* __restrict__ g_base, const float* __restrict__ terms, int64_t per_sample) {
  __shared__ float red[6][256];
  const int64_t n = blockIdx.x;
  float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t i = threadIdx.x; i < per_sample; i += blockDim.x) {
    const float* t = terms + (n * per_sample + i) * 6;
#pragma unroll
    for (int q = 0; q < 6; ++q) acc[q] += t[q];
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) red[q][threadIdx.x] = acc[q];
  __syncthreads();
  for (int half = blockDim.x / 2; half > 0; half >>= 1) {
    if (threadIdx.x < half) {
#pragma unroll
      for (int q = 0; q < 6; ++q) red[q][threadIdx.x] += red[q][threadIdx.x + half];
    }
    __syncthreads();
  }
  if (threadIdx.x < 6) g_base[n * 6 + threadIdx.x] = red[threadIdx.x][0];
}

inline int flow_grid(int64_t total) {
  int64_t g = (total + 255) / 256;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  return static_cast<int>(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace
}  // namespace gg

using namespace gg;

extern "C" {

int gg_flow_compose_forward(float* delta_flow, float* flow, const float* low_flow, const float* mask,
                            const float* identity_flow, const float* base_warp, const float* alpha, int64_t N,
                            int H, int W, int S, void* stream) {
  if (N < 0 || H < 1 || W < 1 || S < 1) return fail(GG_ERR_BAD_ARG, "flow_compose_forward: bad shape");
  if (N == 0) return GG_OK;
  if (!delta_flow || !low_flow || !mask) return fail(GG_ERR_BAD_ARG, "flow_compose_forward: null tensor");
  if (flow && !identity_flow) return fail(GG_ERR_BAD_ARG, "flow_compose_forward: flow output needs identity_flow");
  FlowParams p{N, H, W, S};
  const int64_t total = N * S * S * H * static_cast<int64_t>(W);
  flow_compose_fwd_kernel<<<flow_grid(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      delta_flow, flow, low_flow, mask, identity_flow, base_warp, alpha, p, total);
  GG_CHECK_LAUNCH("flow_compose_fwd launch");
  return GG_OK;
}

int64_t gg_flow_compose_backward_workspace(int64_t N, int H, int W, int S) {
  const int64_t pixels = N * S * S * H * static_cast<int64_t>(W);
  return pixels * 9 * static_cast<int64_t>(sizeof(float2)) + pixels * 6 * static_cast<int64_t>(sizeof(float));
}

int gg_flow_compose_backward(float* grad_mask, float* grad_low_flow, float* grad_base_warp, void* workspace,
                             const float* grad_delta, const float* grad_flow, const float* low_flow, const float* mask,
                             const float* identity_flow, const float* base_warp, const float* alpha, int64_t N,
                             int H, int W, int S, void* stream) {
  if (N < 0 || H < 1 || W < 1 || S < 1) return fail(GG_ERR_BAD_ARG, "flow_compose_backward: bad shape");
  if (N == 0) return GG_OK;
  if (!low_flow || !mask) return fail(GG_ERR_BAD_ARG, "flow_compose_backward: null tensor");
  if (grad_flow && base_warp && !identity_flow) return fail(GG_ERR_BAD_ARG, "flow_compose_backward: identity_flow required");
  FlowParams p{N, H, W, S};
  const int64_t total = N * S * S * H * static_cast<int64_t>(W);
  if ((grad_low_flow || grad_base_warp) && !workspace)
    return fail(GG_ERR_BAD_ARG, "flow_compose_backward: grad_low_flow / grad_base_warp need a workspace");
  auto st = static_cast<cudaStream_t>(stream);
  // both outputs are written in full (the caller need not zero them)
  float2* low_terms = grad_low_flow ? static_cast<float2*>(workspace) : nullptr;
  float* base_terms = (grad_base_warp && grad_flow && base_warp)
                          ? reinterpret_cast<float*>(static_cast<char*>(workspace) + total * 9 * sizeof(float2)) : nullptr;
  if (grad_base_warp && !base_terms) {
    if (cudaMemsetAsync(grad_base_warp, 0, N * 6 * sizeof(float), st) != cudaSuccess)
      return fail(GG_ERR_CUDA, "flow_compose_backward: memset failed");
  }
  flow_compose_bwd_kernel<<<flow_grid(total), 256, 0, st>>>(
      grad_mask, low_terms, base_terms, grad_delta, grad_flow, low_flow, mask, identity_flow, base_warp, alpha,
      p, total);
  GG_CHECK_LAUNCH("flow_compose_bwd launch");
  if (low_terms) {
    const int64_t cells = N * H * static_cast<int64_t>(W);
    flow_low_gather_kernel<<<flow_grid(cells * 32), 256, 0, st>>>(grad_low_flow, low_terms, p, cells);
    GG_CHECK_LAUNCH("flow_low_gather launch");
  }
  if (base_terms) {
    flow_base_reduce_kernel<<<static_cast<unsigned>(N), 256, 0, st>>>(grad_base_warp, base_terms, total / N);
    GG_CHECK_LAUNCH("flow_base_reduce launch");
  }
  return GG_OK;
}

}  // extern "C"
