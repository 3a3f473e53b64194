// warp.cu -- antialiased (mip-mapped) bilinear grid sampling in one pass, forward and backward (sm_100a).
//
// Replaces reference models/spatial_transformers/antialiased_sampling.py:35-238 (MipmapWarp) which issues
// ~30 ATen launches per call, materialises an (N, C, D, H, W) Gaussian *stack* (every level upsampled back
// to full resolution), and synchronises with the host (`levels.max().ceil().item()`, :52) to size it.
// Here the pyramid stays at its native resolutions (levels 1..E, built by mip_down_kernel) and ONE kernel
// per direction evaluates, per output pixel: level of detail from the 4 grid neighbours (:62-97,197-210),
// the two bracketing levels, the bilinear sample of each level *as if* it had been upsampled
// (align_corners=False rules of F.interpolate nested inside those of F.grid_sample, :155-178) and the
// linear blend (:227-237).  No stack, no host sync: levels above the batch maximum simply get weight 0.
// Padding modes zeros/border/reflection follow ATen's grid_sampler (GridSampler.h) exactly, including the
// corner in-bounds tests, so corner/level indices are identical integers.
//
// HBM-bound in principle (algorithmic bytes 4*N*(C*Hs*Ws + C*Ho*Wo + 2*Ho*Wo)) but at GANgealing's sizes
// (3 x 128^2 .. 3 x 512^2 per sample) the whole working set is L2-resident and the win is launch count.
#include "common.cuh"

namespace gg {
namespace {

constexpr int kMaxLevels = 8;  // extra pyramid levels (1..E); MipmapWarp(max_num_levels=8) needs 7

struct Pyramid {
  int hs, ws;            // source size
  int lp;                // reflect padding (left/top) applied before the pyramid when ws is not a power of two
  int hp, wp;            // padded size
  int extra;             // E
  int64_t offset[kMaxLevels + 1];  // float offset of level i (1-based) inside the pyramid buffer
  int64_t planes;
};

inline bool make_pyramid(int hs, int ws, int64_t planes, int extra, Pyramid* p, const char** why) {
  p->hs = hs; p->ws = ws; p->planes = planes; p->extra = extra;
  int lp = 0, rp = 0;
  if (ws > 0 && (ws & (ws - 1)) != 0) {  // antialiased_sampling.py:130-137 (width decides, applied to both axes)
    int target = 1;
    while (target < ws) target <<= 1;
    const int total = target - ws;
    lp = total / 2;
    rp = total - lp;
  }
  p->lp = lp;
  p->hp = hs + lp + rp;
  p->wp = ws + lp + rp;
  if (lp >= hs || rp >= hs || lp >= ws || rp >= ws) { *why = "reflect padding to a power of two exceeds the source size"; return false; }
  if (extra < 0 || extra > kMaxLevels) { *why = "too many mip levels"; return false; }
  int64_t off = 0;
  for (int i = 1; i <= extra; ++i) {
    if ((p->hp >> (i - 1)) < 2 || (p->wp >> (i - 1)) < 2 || (p->hp % (1 << i)) != 0 || (p->wp % (1 << i)) != 0) {
      *why = "source size is not divisible by 2^levels (the reference's Gaussian stack cannot be built either)";
      return false;
    }
    p->offset[i] = off;
    off += planes * (p->hp >> i) * static_cast<int64_t>(p->wp >> i);
  }
  p->offset[0] = off;  // total
  return true;
}

__device__ __forceinline__ int reflect_idx(int j, int size) {  // ReflectionPad semantics (no edge repeat)
  if (j < 0) j = -j;
  if (j >= size) j = 2 * (size - 1) - j;
  return j;
}

// level i (from level i-1): ReflectionPad2d(1) + [1,3,3,1]^2/64 stride 2  (antialiased_sampling.py:111-117)
// SRC_LEVEL: the input is the source image seen through the virtual pow2 reflect padding.
template <typename T, bool SRC_LEVEL>
__global__ void mip_down_kernel(float* __restrict__ out, const T* __restrict__ in, int in_h, int in_w,
                                int src_h, int src_w, int lp, int64_t total) {
  const int oh = in_h >> 1, ow = in_w >> 1;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(idx % ow);
    const int64_t t = idx / ow;
    const int y = static_cast<int>(t % oh);
    const int64_t plane = t / oh;
    const float f[4] = {1.f, 3.f, 3.f, 1.f};
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      int yy = reflect_idx(2 * y + a - 1, in_h);
      if (SRC_LEVEL) yy = reflect_idx(yy - lp, src_h);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        int xx = reflect_idx(2 * x + b - 1, in_w);
        if (SRC_LEVEL) xx = reflect_idx(xx - lp, src_w);
        const int64_t pos = SRC_LEVEL ? (plane * src_h + yy) * static_cast<int64_t>(src_w) + xx
                                      : (plane * in_h + yy) * static_cast<int64_t>(in_w) + xx;
        acc = fmaf(Cvt<T>::to_f(in[pos]), f[a] * f[b] * (1.f / 64.f), acc);
      }
    }
    out[idx] = acc;
  }
}

// adjoint of mip_down_kernel: grad_in += down^T(grad_out)   (atomics: reflected taps overlap)
template <bool SRC_LEVEL>
__global__ void mip_down_bwd_kernel(float* __restrict__ grad_in, const float* __restrict__ grad_out, int in_h,
                                    int in_w, int src_h, int src_w, int lp, int64_t total) {
  const int oh = in_h >> 1, ow = in_w >> 1;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(idx % ow);
    const int64_t t = idx / ow;
    const int y = static_cast<int>(t % oh);
    const int64_t plane = t / oh;
    const float g = grad_out[idx];
    if (g == 0.f) continue;
    const float f[4] = {1.f, 3.f, 3.f, 1.f};
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      int yy = reflect_idx(2 * y + a - 1, in_h);
      if (SRC_LEVEL) yy = reflect_idx(yy - lp, src_h);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        int xx = reflect_idx(2 * x + b - 1, in_w);
        if (SRC_LEVEL) xx = reflect_idx(xx - lp, src_w);
        const int64_t pos = SRC_LEVEL ? (plane * src_h + yy) * static_cast<int64_t>(src_w) + xx
                                      : (plane * in_h + yy) * static_cast<int64_t>(in_w) + xx;
        atomicAdd(grad_in + pos, g * (f[a] * f[b] * (1.f / 64.f)));
      }
    }
  }
}

// ---------------------------------------------------------------- coordinate transforms (ATen GridSampler.h)
struct Coord {
  float x;      // source coordinate after padding-mode handling
  float mult;   // d x / d grid
};

__device__ __forceinline__ Coord reflect_coord(float in, int twice_low, int twice_high) {
  Coord r;
  if (twice_low == twice_high) { r.x = 0.f; r.mult = 0.f; return r; }
  float mult = 1.f;
  const float mn = static_cast<float>(twice_low) / 2.f;
  const float span = static_cast<float>(twice_high - twice_low) / 2.f;
  in = in - mn;
  if (in < 0.f) { mult = -1.f; in = -in; }
  const float extra = fmodf(in, span);
  const int flips = static_cast<int>(floorf(in / span));
  if (flips % 2 == 0) { r.x = extra + mn; r.mult = mult; }
  else { r.x = span - extra + mn; r.mult = -mult; }
  return r;
}

__device__ __forceinline__ Coord source_coord(float g, int size, int pad_mode) {
  Coord c;
  c.x = ((g + 1.f) * size - 1.f) / 2.f;   // align_corners = False
  c.mult = static_cast<float>(size) / 2.f;
  if (pad_mode == GG_PAD_BORDER) {
    // clip_coordinates_set_grad: zero gradient AT and beyond the borders
    if (c.x <= 0.f) { c.x = 0.f; c.mult = 0.f; }
    else if (c.x >= static_cast<float>(size - 1)) { c.x = static_cast<float>(size - 1); c.mult = 0.f; }
  } else if (pad_mode == GG_PAD_REFLECTION) {
    const Coord r = reflect_coord(c.x, -1, 2 * size - 1);
    c.x = r.x; c.mult *= r.mult;
    if (c.x <= 0.f) { c.x = 0.f; c.mult = 0.f; }
    else if (c.x >= static_cast<float>(size - 1)) { c.x = static_cast<float>(size - 1); c.mult = 0.f; }
  }
  return c;
}

// F.interpolate(bilinear, align_corners=False, scale_factor=2^i) source index of destination `dst`
struct Up1D { int i0, i1; float l0, l1; };
__device__ __forceinline__ Up1D upsample_index(int dst, float inv_scale, int in_size) {
  Up1D u;
  float src = (static_cast<float>(dst) + 0.5f) * inv_scale - 0.5f;
  if (src < 0.f) src = 0.f;
  u.i0 = static_cast<int>(src);
  u.i1 = u.i0 + ((u.i0 < in_size - 1) ? 1 : 0);
  u.l1 = src - static_cast<float>(u.i0);
  u.l0 = 1.f - u.l1;
  return u;
}

struct LevelInfo {
  float level;     // after both clamps
  int l0, l1;      // floor / ceil
  float w;         // level % 1
  // gradient bookkeeping
  float dmax;      // max clamped neighbour distance
  int arg;         // 0 left, 1 right, 2 up, 3 down (first maximum)
  float sq_arg;    // unclamped squared distance of the arg-max neighbour
  float dx, dy;    // (other - c) of the arg-max neighbour, LOD coordinates
  bool pass;       // level gradient flows (inside both clamps)
};

// `grid_at(y, x) -> float2`: the sampling grid, read from a tensor or generated on the fly (fused compose)
template <typename GridAt>
__device__ __forceinline__ LevelInfo level_of_detail(GridAt grid_at, int oy, int ox, int ho, int wo,
                                                     int hs, int ws, float max_level, float min_level) {
  // antialiased_sampling.py:181-210 and :62-97
  auto coord = [&](int y, int x, float& cx, float& cy) {
    const float2 g = grid_at(y, x);
    cx = (static_cast<float>(ws) - 1.f) * (g.x + 1.f) / 2.f;
    cy = (static_cast<float>(hs) - 1.f) * (g.y + 1.f) / 2.f;
  };
  float cx, cy;
  coord(oy, ox, cx, cy);
  const int ny[4] = {oy, oy, max(oy - 1, 0), min(oy + 1, ho - 1)};
  const int nx[4] = {max(ox - 1, 0), min(ox + 1, wo - 1), ox, ox};
  LevelInfo li;
  li.dmax = -1.f; li.arg = 0; li.sq_arg = 0.f; li.dx = 0.f; li.dy = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float ox_, oy_;
    coord(ny[k], nx[k], ox_, oy_);
    const float dx = ox_ - cx, dy = oy_ - cy;
    const float sq = dx * dx + dy * dy;
    const float d = sqrtf(fmaxf(sq, 1.f));
    if (d > li.dmax) { li.dmax = d; li.arg = k; li.sq_arg = sq; li.dx = dx; li.dy = dy; }
  }
  const float raw = log2f(li.dmax);
  float lvl = fminf(fmaxf(raw, 0.f), max_level);
  li.pass = (raw >= 0.f) && (raw <= max_level) && (lvl >= min_level);
  lvl = fmaxf(lvl, min_level);
  li.level = lvl;
  const float fl = floorf(lvl);
  li.l0 = static_cast<int>(fl);
  li.l1 = static_cast<int>(ceilf(lvl));
  li.w = lvl - fl;
  return li;
}

struct SampleGeom {   // bilinear corners of one output pixel (shared by all levels and channels)
  int x0, y0;
  float wx0, wx1, wy0, wy1;   // wx1 = ix - x0, wx0 = x1 - ix ...
  bool in_x0, in_x1, in_y0, in_y1;
  float mx, my;               // d ix / d gx, d iy / d gy
};

__device__ __forceinline__ SampleGeom sample_geom(float gx, float gy, int hs, int ws, int pad_mode) {
  SampleGeom s;
  const Coord cx = source_coord(gx, ws, pad_mode);
  const Coord cy = source_coord(gy, hs, pad_mode);
  const float fx = floorf(cx.x), fy = floorf(cy.x);
  s.x0 = static_cast<int>(fx); s.y0 = static_cast<int>(fy);
  s.wx1 = cx.x - fx; s.wx0 = (fx + 1.f) - cx.x;
  s.wy1 = cy.x - fy; s.wy0 = (fy + 1.f) - cy.x;
  s.in_x0 = s.x0 >= 0 && s.x0 < ws; s.in_x1 = s.x0 + 1 >= 0 && s.x0 + 1 < ws;
  s.in_y0 = s.y0 >= 0 && s.y0 < hs; s.in_y1 = s.y0 + 1 >= 0 && s.y0 + 1 < hs;
  s.mx = cx.mult; s.my = cy.mult;
  return s;
}

// value of pyramid level `lev` (>= 1), upsampled to full resolution, at source pixel (y, x)
__device__ __forceinline__ float level_value(const float* __restrict__ lvl_plane, int lh, int lw, float inv_scale,
                                             int y, int x, int lp) {
  const Up1D uy = upsample_index(y + lp, inv_scale, lh);
  const Up1D ux = upsample_index(x + lp, inv_scale, lw);
  const float v00 = lvl_plane[static_cast<int64_t>(uy.i0) * lw + ux.i0];
  const float v01 = lvl_plane[static_cast<int64_t>(uy.i0) * lw + ux.i1];
  const float v10 = lvl_plane[static_cast<int64_t>(uy.i1) * lw + ux.i0];
  const float v11 = lvl_plane[static_cast<int64_t>(uy.i1) * lw + ux.i1];
  return uy.l0 * (ux.l0 * v00 + ux.l1 * v01) + uy.l1 * (ux.l0 * v10 + ux.l1 * v11);
}

struct WarpParams {
  int64_t n; int c; int hs, ws, ho, wo;
  int pad_mode;
  float max_level, min_level;
  int lp, hp, wp, extra;
  int64_t offset[kMaxLevels + 1];
};

// bilinear sample of level `lev` for channel plane; returns value and (optionally) d/dix, d/diy
template <typename T, bool GRAD>
__device__ __forceinline__ float sample_level(const T* __restrict__ src_plane, const float* __restrict__ pyr,
                                              const WarpParams& p, int64_t plane, int lev, const SampleGeom& s,
                                              float* dix, float* diy) {
  float v[2][2];
  const float* lvl_plane = nullptr;
  int lh = 0, lw = 0;
  float inv = 1.f;
  if (lev > 0) {
    lh = p.hp >> lev; lw = p.wp >> lev;
    lvl_plane = pyr + p.offset[lev] + plane * lh * static_cast<int64_t>(lw);
    inv = 1.f / static_cast<float>(1 << lev);
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const bool ok = (a ? s.in_y1 : s.in_y0) && (b ? s.in_x1 : s.in_x0);
      float val = 0.f;
      if (ok) {
        const int y = s.y0 + a, x = s.x0 + b;
        val = (lev == 0) ? Cvt<T>::to_f(src_plane[static_cast<int64_t>(y) * p.ws + x])
                         : level_value(lvl_plane, lh, lw, inv, y, x, p.lp);
      }
      v[a][b] = val;
    }
  if (GRAD) {
    // ATen grid_sampler_2d_backward: gix -= nw*(iy_se - iy) ... with our weights
    *dix = -v[0][0] * s.wy0 + v[0][1] * s.wy0 - v[1][0] * s.wy1 + v[1][1] * s.wy1;
    *diy = -v[0][0] * s.wx0 - v[0][1] * s.wx1 + v[1][0] * s.wx0 + v[1][1] * s.wx1;
  }
  return v[0][0] * (s.wx0 * s.wy0) + v[0][1] * (s.wx1 * s.wy0) + v[1][0] * (s.wx0 * s.wy1) + v[1][1] * (s.wx1 * s.wy1);
}

template <typename T, bool MIP>
__global__ void __launch_bounds__(256)
warp_fwd_kernel(T* __restrict__ out, float* __restrict__ levels_out, const T* __restrict__ src,
                const float* __restrict__ pyr, const float* __restrict__ grid, const __grid_constant__ WarpParams p,
                int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(idx % p.wo);
    const int64_t t = idx / p.wo;
    const int oy = static_cast<int>(t % p.ho);
    const int64_t n = t / p.ho;
    const float* grid_n = grid + n * p.ho * static_cast<int64_t>(p.wo) * 2;
    const float2 g = *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(oy) * p.wo + ox) * 2);
    const SampleGeom s = sample_geom(g.x, g.y, p.hs, p.ws, p.pad_mode);
    int l0 = 0, l1 = 0;
    float w = 0.f;
    if (MIP) {
      auto grid_at = [&](int y, int x) { return *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(y) * p.wo + x) * 2); };
      const LevelInfo li = level_of_detail(grid_at, oy, ox, p.ho, p.wo, p.hs, p.ws, p.max_level, p.min_level);
      l0 = li.l0; l1 = li.l1; w = li.w;
      if (levels_out) levels_out[idx] = li.level;
    }
    for (int c = 0; c < p.c; ++c) {
      const int64_t plane = n * p.c + c;
      const T* src_plane = src + plane * p.hs * static_cast<int64_t>(p.ws);
      const float o0 = sample_level<T, false>(src_plane, pyr, p, plane, l0, s, nullptr, nullptr);
      float o = o0;
      if (MIP && l1 != l0) {
        const float o1 = sample_level<T, false>(src_plane, pyr, p, plane, l1, s, nullptr, nullptr);
        o = o0 + w * (o1 - o0);
      }
      out[(plane * p.ho + oy) * static_cast<int64_t>(p.wo) + ox] = Cvt<T>::from_f(o);
    }
  }
}

// ---------------------------------------------------------------- integer work of the sampler, exported for exact tests
// One int4 per output pixel: (x0, y0) = the north-west bilinear corner in source pixels after the padding-mode transform
// (ATen grid_sampler's floor(ix), floor(iy)), and (l0, l1) = floor / ceil of the level of detail -- produced by the SAME
// device functions (sample_geom, level_of_detail) the sampling kernels call, so the parity tests can compare the integers
// themselves with the oracle's (oracle/sampling.py grid_sample_bilinear / mipmap_warp_ref) instead of inferring them.
__global__ void __launch_bounds__(256)
sample_indices_kernel(int4* __restrict__ out, const float* __restrict__ grid, const __grid_constant__ WarpParams p, int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(idx % p.wo);
    const int64_t t = idx / p.wo;
    const int oy = static_cast<int>(t % p.ho);
    const int64_t n = t / p.ho;
    const float* grid_n = grid + n * p.ho * static_cast<int64_t>(p.wo) * 2;
    const float2 g = *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(oy) * p.wo + ox) * 2);
    const SampleGeom s = sample_geom(g.x, g.y, p.hs, p.ws, p.pad_mode);
    auto grid_at = [&](int y, int x) { return *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(y) * p.wo + x) * 2); };
    const LevelInfo li = level_of_detail(grid_at, oy, ox, p.ho, p.wo, p.hs, p.ws, p.max_level, p.min_level);
    out[idx] = make_int4(s.x0, s.y0, li.l0, li.l1);
  }
}

// ---------------------------------------------------------------- the STN's sampling in ONE pass
// north_star: "the STN's antialiased bilinear grid_sample fused with flow-compose in one pass".  The sampling grid is never
// read from memory: every output pixel GENERATES its coordinate (and those of its 4 neighbours, for the level of detail)
// from the head's raw regression outputs --
//   MODE 1 (SimilarityHead, warping_heads.py:120-136): F.affine_grid(theta, align_corners=False): g = theta . [x, y, 1],
//           x = (2*ox + 1)/Wo - 1
//   MODE 2 (FlowHead, warping_heads.py:180-193,239-244,268-277): RAFT convex up-sampling (softmax over 9 mask logits x the 3x3
//           neighbourhood of s*low_flow) + identity + apply_affine(base_warp) + alpha lerp
// and then runs the level-of-detail / trilinear sampling of warp_fwd_kernel.  The grid (and the residual flow the TV
// regulariser needs) are WRITTEN as by-products (the callers return them), replacing affine_grid (a bmm + 3 elementwise
// launches) or the separate flow_compose pass and the grid read-back.
struct ComposeParams {
  const float* theta;     // MODE 1: (N, 2, 3) sampling matrices.  MODE 2: base warp (N, 2, 3) or null
  const float* low;       // MODE 2: (N, lh, lw, 2)
  const float* mask;      // MODE 2: (N, 9*s*s, lh, lw)
  const float* identity;  // MODE 2: (s*lh, s*lw, 2) identity sampling grid (the head's buffer)
  const float* alpha;     // MODE 2: (N) or null
  int lh, lw, s;
  float* grid_out;        // (N, Ho, Wo, 2) or null
  float* delta_out;       // MODE 2: (N, Ho, Wo, 2) or null
};

template <int MODE>
__device__ __forceinline__ float2 compose_at(const ComposeParams& cp, const WarpParams& p, int64_t n, int y, int x,
                                             float2* delta) {
  if (MODE == 1) {
    const float* M = cp.theta + n * 6;
    const float bx = (2.f * static_cast<float>(x) + 1.f) / static_cast<float>(p.wo) - 1.f;
    const float by = (2.f * static_cast<float>(y) + 1.f) / static_cast<float>(p.ho) - 1.f;
    return make_float2(fmaf(M[0], bx, fmaf(M[1], by, M[2])), fmaf(M[3], bx, fmaf(M[4], by, M[5])));
  } else {
    const int h = y / cp.s, w = x / cp.s, sy = y - h * cp.s, sx = x - w * cp.s;
    float lg[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      lg[k] = __ldg(cp.mask + ((((n * 9 + k) * cp.s + sy) * cp.s + sx) * cp.lh + h) * static_cast<int64_t>(cp.lw) + w);
      mx = fmaxf(mx, lg[k]);
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { lg[k] = expf(lg[k] - mx); sum += lg[k]; }
    const float inv = 1.f / sum;
    float dx = 0.f, dy = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int hh = h + k / 3 - 1, ww = w + k % 3 - 1;
      if (hh >= 0 && hh < cp.lh && ww >= 0 && ww < cp.lw) {
        const float2 f = __ldg(reinterpret_cast<const float2*>(cp.low + ((n * cp.lh + hh) * static_cast<int64_t>(cp.lw) + ww) * 2));
        const float pk = lg[k] * inv;
        dx = fmaf(pk, static_cast<float>(cp.s) * f.x, dx);
        dy = fmaf(pk, static_cast<float>(cp.s) * f.y, dy);
      }
    }
    if (delta) *delta = make_float2(dx, dy);
    const float2 id = __ldg(reinterpret_cast<const float2*>(cp.identity + (static_cast<int64_t>(y) * p.wo + x) * 2));
    float gx = id.x + dx, gy = id.y + dy;
    if (cp.theta) {
      const float* M = cp.theta + n * 6;
      const float tx = M[0] * gx + M[1] * gy + M[2];
      const float ty = M[3] * gx + M[4] * gy + M[5];
      gx = tx; gy = ty;
    }
    if (cp.alpha) {
      const float a = __ldg(cp.alpha + n);
      gx = id.x + a * (gx - id.x);
      gy = id.y + a * (gy - id.y);
    }
    return make_float2(gx, gy);
  }
}

// CTA = a 32 x 8 tile of output pixels of one sample.  Every thread generates the coordinate of ITS pixel once and parks it
// in shared memory together with the one-pixel halo (computed by the first 84 threads), so the level of detail reads its 4
// neighbours from shared memory instead of regenerating them (5x fewer softmax evaluations than a per-thread recompute).
constexpr int kTileX = 32, kTileY = 8;

template <typename T, bool MIP, int MODE>
__global__ void __launch_bounds__(kTileX * kTileY)
warp_compose_fwd_kernel(T* __restrict__ out, float* __restrict__ levels_out, const T* __restrict__ src,
                        const float* __restrict__ pyr, const ComposeParams cp, const __grid_constant__ WarpParams p,
                        int tiles_x, int tiles_y) {
  __shared__ float2 tile[kTileY + 2][kTileX + 2];
  const int tx = threadIdx.x % kTileX, ty = threadIdx.x / kTileX;
  const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y;
  const int64_t n = blockIdx.x / (tiles_x * tiles_y);
  const int x0 = bx * kTileX, y0 = by * kTileY;
  const int ox = x0 + tx, oy = y0 + ty;
  const bool live = ox < p.wo && oy < p.ho;
  float2 delta = make_float2(0.f, 0.f);
  float2 g = make_float2(0.f, 0.f);
  if (live) {
    g = compose_at<MODE>(cp, p, n, oy, ox, &delta);
    const int64_t idx = (n * p.ho + oy) * static_cast<int64_t>(p.wo) + ox;
    if (cp.grid_out) *reinterpret_cast<float2*>(cp.grid_out + idx * 2) = g;
    if (MODE == 2 && cp.delta_out) *reinterpret_cast<float2*>(cp.delta_out + idx * 2) = delta;
  }
  tile[ty + 1][tx + 1] = g;
  if (MIP) {
    // halo ring: 2*(kTileX + 2) + 2*kTileY = 84 positions, replicate-clamped to the image like the reference's neighbours
    constexpr int kRing = 2 * (kTileX + 2) + 2 * kTileY;
    if (threadIdx.x < kRing) {
      int hy, hx;
      const int r = threadIdx.x;
      if (r < kTileX + 2) { hy = -1; hx = r - 1; }
      else if (r < 2 * (kTileX + 2)) { hy = kTileY; hx = r - (kTileX + 2) - 1; }
      else if (r < 2 * (kTileX + 2) + kTileY) { hy = r - 2 * (kTileX + 2); hx = -1; }
      else { hy = r - 2 * (kTileX + 2) - kTileY; hx = kTileX; }
      const int yy = min(max(y0 + hy, 0), p.ho - 1), xx = min(max(x0 + hx, 0), p.wo - 1);
      tile[hy + 1][hx + 1] = compose_at<MODE>(cp, p, n, yy, xx, nullptr);
    }
    __syncthreads();
  }
  if (!live) return;
  const int64_t idx = (n * p.ho + oy) * static_cast<int64_t>(p.wo) + ox;
  const SampleGeom s = sample_geom(g.x, g.y, p.hs, p.ws, p.pad_mode);
  int l0 = 0, l1 = 0;
  float w = 0.f;
  if (MIP) {
    // (y, x) is replicate-clamped by the caller: a clamped neighbour of an edge pixel is the pixel itself or its in-tile
    // neighbour; positions beyond the image but inside the tile hold clamped coordinates as well (computed above)
    auto grid_at = [&](int y, int x) { return tile[y - y0 + 1][x - x0 + 1]; };
    const LevelInfo li = level_of_detail(grid_at, oy, ox, p.ho, p.wo, p.hs, p.ws, p.max_level, p.min_level);
    l0 = li.l0; l1 = li.l1; w = li.w;
    if (levels_out) levels_out[idx] = li.level;
  }
  for (int c = 0; c < p.c; ++c) {
    const int64_t plane = n * p.c + c;
    const T* src_plane = src + plane * p.hs * static_cast<int64_t>(p.ws);
    const float o0 = sample_level<T, false>(src_plane, pyr, p, plane, l0, s, nullptr, nullptr);
    float o = o0;
    if (MIP && l1 != l0) {
      const float o1 = sample_level<T, false>(src_plane, pyr, p, plane, l1, s, nullptr, nullptr);
      o = o0 + w * (o1 - o0);
    }
    out[(plane * p.ho + oy) * static_cast<int64_t>(p.wo) + ox] = Cvt<T>::from_f(o);
  }
}

// ---------------------------------------------------------------- all pyramid levels in ONE launch
// One CTA per image plane: level 1 is computed from the source (global / L2) into shared memory, every further level from
// the previous one in shared memory; each level is also written to the pyramid buffer.  Used when levels 1..E of a plane
// fit in shared memory (sources up to ~384^2); larger sources take one mip_down launch per level.
template <typename T>
__global__ void __launch_bounds__(512)
mip_build_all_kernel(float* __restrict__ pyr, const T* __restrict__ src, const __grid_constant__ Pyramid py) {
  extern __shared__ float lv[];               // levels 1..E back to back
  const int64_t plane = blockIdx.x;
  const float f[4] = {1.f, 3.f, 3.f, 1.f};
  int sm_off = 0, prev_off = 0;
  for (int i = 1; i <= py.extra; ++i) {
    const int in_h = py.hp >> (i - 1), in_w = py.wp >> (i - 1);
    const int oh = in_h >> 1, ow = in_w >> 1;
    float* dst = lv + sm_off;
    const float* prev = lv + prev_off;
    float* gout = pyr + py.offset[i] + plane * oh * static_cast<int64_t>(ow);
    for (int o = threadIdx.x; o < oh * ow; o += blockDim.x) {
      const int y = o / ow, x = o - y * ow;
      float acc = 0.f;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        int yy = reflect_idx(2 * y + a - 1, in_h);
        if (i == 1) yy = reflect_idx(yy - py.lp, py.hs);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          int xx = reflect_idx(2 * x + b - 1, in_w);
          float v;
          if (i == 1) {
            xx = reflect_idx(xx - py.lp, py.ws);
            v = Cvt<T>::to_f(src[(plane * py.hs + yy) * static_cast<int64_t>(py.ws) + xx]);
          } else {
            v = prev[yy * in_w + xx];
          }
          acc = fmaf(v, f[a] * f[b] * (1.f / 64.f), acc);
        }
      }
      dst[o] = acc;
      gout[o] = acc;
    }
    __syncthreads();
    prev_off = sm_off;
    sm_off += oh * ow;
  }
}

// scatter `g` (gradient w.r.t. the bilinear sample of level `lev`) into grad_src / grad_pyr
__device__ __forceinline__ void scatter_level(float* __restrict__ grad_src, float* __restrict__ grad_pyr,
                                              const WarpParams& p, int64_t plane, int lev, const SampleGeom& s, float g) {
  if (g == 0.f) return;
  int lh = 0, lw = 0;
  float inv = 1.f;
  float* lvl_plane = nullptr;
  if (lev > 0) {
    lh = p.hp >> lev; lw = p.wp >> lev;
    lvl_plane = grad_pyr + p.offset[lev] + plane * lh * static_cast<int64_t>(lw);
    inv = 1.f / static_cast<float>(1 << lev);
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const bool ok = (a ? s.in_y1 : s.in_y0) && (b ? s.in_x1 : s.in_x0);
      if (!ok) continue;
      const float wt = (a ? s.wy1 : s.wy0) * (b ? s.wx1 : s.wx0) * g;
      const int y = s.y0 + a, x = s.x0 + b;
      if (lev == 0) {
        atomicAdd(grad_src + (plane * p.hs + y) * static_cast<int64_t>(p.ws) + x, wt);
      } else {
        const Up1D uy = upsample_index(y + p.lp, inv, lh);
        const Up1D ux = upsample_index(x + p.lp, inv, lw);
        atomicAdd(lvl_plane + static_cast<int64_t>(uy.i0) * lw + ux.i0, wt * uy.l0 * ux.l0);
        atomicAdd(lvl_plane + static_cast<int64_t>(uy.i0) * lw + ux.i1, wt * uy.l0 * ux.l1);
        atomicAdd(lvl_plane + static_cast<int64_t>(uy.i1) * lw + ux.i0, wt * uy.l1 * ux.l0);
        atomicAdd(lvl_plane + static_cast<int64_t>(uy.i1) * lw + ux.i1, wt * uy.l1 * ux.l1);
      }
    }
}

// the level-of-detail part of a grid pixel's gradient that belongs to the neighbour `target` (-1: none)
struct NbGrad {
  float x, y;
  int target, pad;
};

// grad_grid (written in full): each pixel stores its own part; with MIP the part owed to a neighbour goes to `nb` (the
// caller's workspace), and warp_grid_gather_kernel adds it in a fixed order (no float atomics: the same bits on every run)
template <typename T, bool MIP>
__global__ void __launch_bounds__(256)
warp_bwd_kernel(float* __restrict__ grad_src, float* __restrict__ grad_pyr, float* __restrict__ grad_grid,
                NbGrad* __restrict__ nb, const T* __restrict__ grad_out, const T* __restrict__ src,
                const float* __restrict__ pyr, const float* __restrict__ grid, const __grid_constant__ WarpParams p,
                int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(idx % p.wo);
    const int64_t t = idx / p.wo;
    const int oy = static_cast<int>(t % p.ho);
    const int64_t n = t / p.ho;
    const int64_t grid_off = n * p.ho * static_cast<int64_t>(p.wo) * 2;
    const float* grid_n = grid + grid_off;
    const float2 g = *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(oy) * p.wo + ox) * 2);
    const SampleGeom s = sample_geom(g.x, g.y, p.hs, p.ws, p.pad_mode);
    LevelInfo li;
    li.l0 = li.l1 = 0; li.w = 0.f; li.pass = false;
    if (MIP) {
      auto grid_at = [&](int y, int x) { return *reinterpret_cast<const float2*>(grid_n + (static_cast<int64_t>(y) * p.wo + x) * 2); };
      li = level_of_detail(grid_at, oy, ox, p.ho, p.wo, p.hs, p.ws, p.max_level, p.min_level);
    }
    float gix = 0.f, giy = 0.f, glevel = 0.f;
    for (int c = 0; c < p.c; ++c) {
      const int64_t plane = n * p.c + c;
      const float go = Cvt<T>::to_f(grad_out[(plane * p.ho + oy) * static_cast<int64_t>(p.wo) + ox]);
      const T* src_plane = src + plane * p.hs * static_cast<int64_t>(p.ws);
      float dx0 = 0.f, dy0 = 0.f, dx1 = 0.f, dy1 = 0.f;
      const bool two = MIP && (li.l1 != li.l0);
      if (grad_grid) {
        const float o0 = sample_level<T, true>(src_plane, pyr, p, plane, li.l0, s, &dx0, &dy0);
        float k0 = 1.f;
        if (two) {
          const float o1 = sample_level<T, true>(src_plane, pyr, p, plane, li.l1, s, &dx1, &dy1);
          k0 = 1.f - li.w;
          glevel += go * (o1 - o0);
        }
        gix += go * (k0 * dx0 + (two ? li.w * dx1 : 0.f));
        giy += go * (k0 * dy0 + (two ? li.w * dy1 : 0.f));
      }
      if (grad_src) {
        scatter_level(grad_src, grad_pyr, p, plane, li.l0, s, go * (two ? 1.f - li.w : 1.f));
        if (two) scatter_level(grad_src, grad_pyr, p, plane, li.l1, s, go * li.w);
      }
    }
    if (grad_grid) {
      float* gg_n = grad_grid + grid_off;
      float ax = gix * s.mx, ay = giy * s.my;
      NbGrad out_nb{0.f, 0.f, -1, 0};
      if (MIP && li.pass && glevel != 0.f && li.sq_arg >= 1.f) {
        // level = log2(dmax); dmax = sqrt(sq) of the arg-max neighbour (clamp(min=1) passes: sq >= 1)
        const float g_sq = glevel / (li.dmax * 0.6931471805599453f) * (0.5f / li.dmax);
        const float sx = (static_cast<float>(p.ws) - 1.f) * 0.5f, sy = (static_cast<float>(p.hs) - 1.f) * 0.5f;
        const float gox = 2.f * li.dx * g_sq * sx, goy = 2.f * li.dy * g_sq * sy;
        const int ny = (li.arg == 2) ? max(oy - 1, 0) : (li.arg == 3 ? min(oy + 1, p.ho - 1) : oy);
        const int nx = (li.arg == 0) ? max(ox - 1, 0) : (li.arg == 1 ? min(ox + 1, p.wo - 1) : ox);
        out_nb = NbGrad{gox, goy, ny * p.wo + nx, 0};
        ax -= gox; ay -= goy;
      }
      *reinterpret_cast<float2*>(gg_n + (static_cast<int64_t>(oy) * p.wo + ox) * 2) = make_float2(ax, ay);
      if (MIP) nb[idx] = out_nb;
    }
  }
}

// grad_grid[pixel] += the parts its neighbours (and, clamped at a border, itself) owe it, in a fixed order
__global__ void __launch_bounds__(256)
warp_grid_gather_kernel(float* __restrict__ grad_grid, const NbGrad* __restrict__ nb, int ho, int wo, int64_t total) {
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(idx % wo);
    const int oy = static_cast<int>((idx / wo) % ho);
    const int me = oy * wo + ox;
    const int64_t base = idx - me;
    float gx = 0.f, gy = 0.f;
    const int dy[5] = {0, 0, 0, -1, 1}, dx[5] = {0, -1, 1, 0, 0};
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      const int y = oy + dy[q], x = ox + dx[q];
      if (y < 0 || y >= ho || x < 0 || x >= wo) continue;
      const NbGrad v = nb[base + y * wo + x];
      if (v.target == me) { gx += v.x; gy += v.y; }
    }
    float2* g = reinterpret_cast<float2*>(grad_grid + idx * 2);
    float2 cur = *g;
    cur.x += gx; cur.y += gy;
    *g = cur;
  }
}

inline int grid_for(int64_t total, int threads) {
  int64_t g = (total + threads - 1) / threads;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  return static_cast<int>(g < cap ? (g > 0 ? g : 1) : cap);
}

inline int fill_params(WarpParams* wp, int64_t n, int c, int hs, int ws, int ho, int wo, int pad_mode, int extra,
                       float max_level, float min_level) {
  if (n < 0 || c < 0 || hs < 1 || ws < 1 || ho < 0 || wo < 0) return fail(GG_ERR_BAD_ARG, "mipmap_warp: bad shape");
  if (pad_mode < 0 || pad_mode > 2) return fail(GG_ERR_BAD_ARG, "mipmap_warp: padding mode must be 0/1/2");
  Pyramid py;
  const char* why = "";
  if (!make_pyramid(hs, ws, n * c, extra, &py, &why)) return fail(GG_ERR_UNSUPPORTED, "mipmap_warp: %s", why);
  if (extra > 0 && (ceilf(max_level) > extra || ceilf(min_level) > extra))
    return fail(GG_ERR_BAD_ARG, "mipmap_warp: pyramid has %d extra levels but levels up to %g are requested", extra,
                fmaxf(max_level, min_level));
  wp->n = n; wp->c = c; wp->hs = hs; wp->ws = ws; wp->ho = ho; wp->wo = wo; wp->pad_mode = pad_mode;
  wp->max_level = max_level; wp->min_level = min_level;
  wp->lp = py.lp; wp->hp = py.hp; wp->wp = py.wp; wp->extra = extra;
  for (int i = 0; i <= kMaxLevels; ++i) wp->offset[i] = (i <= extra) ? py.offset[i] : 0;
  return GG_OK;
}

template <typename T>
int build_t(float* pyr, const void* src, const Pyramid& py, cudaStream_t st) {
  int64_t sm_floats = 0;
  for (int i = 1; i <= py.extra; ++i) sm_floats += static_cast<int64_t>(py.hp >> i) * (py.wp >> i);
  if (py.extra >= 1 && sm_floats * 4 <= 200 * 1024 && py.planes <= 0x7fffffffLL) {
    const size_t smem = static_cast<size_t>(sm_floats) * sizeof(float);
    if (smem > 48 * 1024) {
      static DeviceOnce configured;
      if (configured.needed()) {
        const cudaError_t e = cudaFuncSetAttribute(mip_build_all_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return cuda_fail(e, "mip_build_all smem opt-in");
        configured.done();
      }
    }
    mip_build_all_kernel<T><<<static_cast<unsigned>(py.planes), 512, smem, st>>>(pyr, static_cast<const T*>(src), py);
    GG_CHECK_LAUNCH("mip_build_all launch");
    return GG_OK;
  }
  for (int i = 1; i <= py.extra; ++i) {
    const int in_h = py.hp >> (i - 1), in_w = py.wp >> (i - 1);
    const int64_t total = py.planes * (in_h >> 1) * static_cast<int64_t>(in_w >> 1);
    if (total == 0) continue;
    float* out = pyr + py.offset[i];
    if (i == 1)
      mip_down_kernel<T, true><<<grid_for(total, 256), 256, 0, st>>>(out, static_cast<const T*>(src), in_h, in_w,
                                                                    py.hs, py.ws, py.lp, total);
    else
      mip_down_kernel<float, false><<<grid_for(total, 256), 256, 0, st>>>(out, pyr + py.offset[i - 1], in_h, in_w,
                                                                         py.hs, py.ws, py.lp, total);
    GG_CHECK_LAUNCH("mip_down launch");
  }
  return GG_OK;
}

}  // namespace
}  // namespace gg

using namespace gg;

extern "C" {

int64_t gg_mipmap_pyramid_elems(int64_t planes, int hs, int ws, int extra_levels) {
  Pyramid py;
  const char* why = "";
  if (planes < 0 || hs < 1 || ws < 1 || !make_pyramid(hs, ws, planes, extra_levels, &py, &why)) return -1;
  return py.offset[0];
}

int gg_mipmap_build(float* pyramid, const void* src, int dtype, int64_t planes, int hs, int ws, int extra_levels,
                    void* stream) {
  Pyramid py;
  const char* why = "";
  if (planes < 0 || hs < 1 || ws < 1) return fail(GG_ERR_BAD_ARG, "mipmap_build: bad shape");
  if (!make_pyramid(hs, ws, planes, extra_levels, &py, &why)) return fail(GG_ERR_UNSUPPORTED, "mipmap_build: %s", why);
  if (planes == 0 || extra_levels == 0) return GG_OK;
  if (!pyramid || !src) return fail(GG_ERR_BAD_ARG, "mipmap_build: null tensor");
  auto st = static_cast<cudaStream_t>(stream);
  switch (dtype) {
    case GG_F32: return build_t<float>(pyramid, src, py, st);
    case GG_F16: return build_t<__half>(pyramid, src, py, st);
    case GG_BF16: return build_t<__nv_bfloat16>(pyramid, src, py, st);
    default: return fail(GG_ERR_UNSUPPORTED, "mipmap_build: dtype %d not supported", dtype);
  }
}

int gg_mipmap_build_backward(float* grad_src, float* grad_pyramid, int64_t planes, int hs, int ws, int extra_levels,
                             void* stream) {
  Pyramid py;
  const char* why = "";
  if (planes < 0 || hs < 1 || ws < 1) return fail(GG_ERR_BAD_ARG, "mipmap_build_backward: bad shape");
  if (!make_pyramid(hs, ws, planes, extra_levels, &py, &why)) return fail(GG_ERR_UNSUPPORTED, "mipmap_build_backward: %s", why);
  if (planes == 0 || extra_levels == 0) return GG_OK;
  if (!grad_src || !grad_pyramid) return fail(GG_ERR_BAD_ARG, "mipmap_build_backward: null tensor");
  auto st = static_cast<cudaStream_t>(stream);
  for (int i = py.extra; i >= 1; --i) {  // coarse to fine: grad_{i-1} += down^T(grad_i)
    const int in_h = py.hp >> (i - 1), in_w = py.wp >> (i - 1);
    const int64_t total = py.planes * (in_h >> 1) * static_cast<int64_t>(in_w >> 1);
    const float* go = grad_pyramid + py.offset[i];
    if (i == 1)
      mip_down_bwd_kernel<true><<<grid_for(total, 256), 256, 0, st>>>(grad_src, go, in_h, in_w, py.hs, py.ws, py.lp, total);
    else
      mip_down_bwd_kernel<false><<<grid_for(total, 256), 256, 0, st>>>(grad_pyramid + py.offset[i - 1], go, in_h, in_w,
                                                                       py.hs, py.ws, py.lp, total);
    GG_CHECK_LAUNCH("mip_down_bwd launch");
  }
  return GG_OK;
}

int gg_warp_sample_indices(int32_t* indices, const float* grid, int64_t N, int hs, int ws, int ho, int wo,
                           float max_level, float min_level, int padding_mode, void* stream) {
  WarpParams wp;
  int rc = fill_params(&wp, N, 1, hs, ws, ho, wo, padding_mode, 0, max_level, min_level);
  if (rc != GG_OK) return rc;
  const int64_t total = N * ho * static_cast<int64_t>(wo);
  if (total == 0) return GG_OK;
  if (!indices || !grid) return fail(GG_ERR_BAD_ARG, "warp_sample_indices: null tensor");
  if (reinterpret_cast<uintptr_t>(indices) & 15) return fail(GG_ERR_BAD_ARG, "warp_sample_indices: indices must be 16-byte aligned");
  sample_indices_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<int4*>(indices), grid, wp, total);
  GG_CHECK_LAUNCH("sample_indices launch");
  return GG_OK;
}

int gg_mipmap_warp_forward(void* out, float* levels_out, const void* src, const float* pyramid, const float* grid,
                           int dtype, int64_t N, int C, int hs, int ws, int ho, int wo, int extra_levels,
                           float max_level, float min_level, int padding_mode, void* stream) {
  WarpParams wp;
  int rc = fill_params(&wp, N, C, hs, ws, ho, wo, padding_mode, extra_levels, max_level, min_level);
  if (rc != GG_OK) return rc;
  const int64_t total = N * ho * static_cast<int64_t>(wo);
  if (total == 0) return GG_OK;
  // C == 0 still writes levels_out: the level of detail depends on the grid alone (out and src are then empty)
  if ((C > 0 && (!out || !src)) || !grid || (extra_levels > 0 && !pyramid))
    return fail(GG_ERR_BAD_ARG, "mipmap_warp_forward: null tensor");
  auto st = static_cast<cudaStream_t>(stream);
  const int gridsz = grid_for(total, 256);
#define GG_FWD(T_)                                                                                               \
  if (extra_levels > 0)                                                                                          \
    warp_fwd_kernel<T_, true><<<gridsz, 256, 0, st>>>(static_cast<T_*>(out), levels_out, static_cast<const T_*>(src), \
                                                      pyramid, grid, wp, total);                               \
  else                                                                                                           \
    warp_fwd_kernel<T_, false><<<gridsz, 256, 0, st>>>(static_cast<T_*>(out), levels_out, static_cast<const T_*>(src), \
                                                       pyramid, grid, wp, total)
  switch (dtype) {
    case GG_F32: GG_FWD(float); break;
    case GG_F16: GG_FWD(__half); break;
    case GG_BF16: GG_FWD(__nv_bfloat16); break;
    default: return fail(GG_ERR_UNSUPPORTED, "mipmap_warp_forward: dtype %d not supported", dtype);
  }
#undef GG_FWD
  GG_CHECK_LAUNCH("warp_fwd launch");
  return GG_OK;
}

int gg_stn_sample_forward(void* out, float* grid_out, float* delta_out, float* levels_out, const void* src,
                          const float* pyramid, const float* theta, const float* low, const float* mask,
                          const float* identity, const float* alpha, int mode, int dtype, int64_t N, int C, int hs, int ws,
                          int ho, int wo, int lh, int lw, int s, int extra_levels, float max_level, float min_level,
                          int padding_mode, void* stream) {
  WarpParams wp;
  int rc = fill_params(&wp, N, C, hs, ws, ho, wo, padding_mode, extra_levels, max_level, min_level);
  if (rc != GG_OK) return rc;
  if (mode != 1 && mode != 2) return fail(GG_ERR_BAD_ARG, "stn_sample: mode must be 1 (affine) or 2 (flow)");
  const int64_t total = N * ho * static_cast<int64_t>(wo);
  if (total == 0) return GG_OK;
  // C == 0 still writes grid_out, delta_out and levels_out, which do not depend on the image (out and src are then empty)
  if ((C > 0 && (!out || !src)) || (extra_levels > 0 && !pyramid)) return fail(GG_ERR_BAD_ARG, "stn_sample: null tensor");
  if (mode == 1 && !theta) return fail(GG_ERR_BAD_ARG, "stn_sample: affine mode needs theta");
  if (mode == 2) {
    if (!low || !mask || !identity) return fail(GG_ERR_BAD_ARG, "stn_sample: flow mode needs low, mask and identity");
    if (s < 1 || lh < 1 || lw < 1 || lh * s != ho || lw * s != wo)
      return fail(GG_ERR_BAD_ARG, "stn_sample: the flow grid (%d x %d, x%d) must match the output size (%d x %d)", lh, lw, s, ho, wo);
  }
  ComposeParams cp;
  cp.theta = theta; cp.low = low; cp.mask = mask; cp.identity = identity; cp.alpha = alpha;
  cp.lh = lh; cp.lw = lw; cp.s = s; cp.grid_out = grid_out; cp.delta_out = delta_out;
  auto st = static_cast<cudaStream_t>(stream);
  const int tiles_x = (wo + kTileX - 1) / kTileX, tiles_y = (ho + kTileY - 1) / kTileY;
  const int64_t ctas = N * tiles_x * static_cast<int64_t>(tiles_y);
  if (ctas > 0x7fffffffLL) return fail(GG_ERR_BAD_ARG, "stn_sample: too many tiles");
  const unsigned gridsz = static_cast<unsigned>(ctas);
#define GG_SS(T_, MIP_, MODE_)                                                                                   \
  warp_compose_fwd_kernel<T_, MIP_, MODE_><<<gridsz, kTileX * kTileY, 0, st>>>(static_cast<T_*>(out), levels_out, \
                                                                 static_cast<const T_*>(src), pyramid, cp, wp, tiles_x, tiles_y)
#define GG_SS_T(T_)                                                                       \
  if (extra_levels > 0) { if (mode == 1) GG_SS(T_, true, 1); else GG_SS(T_, true, 2); }   \
  else { if (mode == 1) GG_SS(T_, false, 1); else GG_SS(T_, false, 2); }
  switch (dtype) {
    case GG_F32: GG_SS_T(float); break;
    case GG_F16: GG_SS_T(__half); break;
    case GG_BF16: GG_SS_T(__nv_bfloat16); break;
    default: return fail(GG_ERR_UNSUPPORTED, "stn_sample: dtype %d not supported", dtype);
  }
#undef GG_SS_T
#undef GG_SS
  GG_CHECK_LAUNCH("warp_compose_fwd launch");
  return GG_OK;
}

int64_t gg_mipmap_warp_backward_workspace(int64_t N, int ho, int wo) {
  return N * ho * static_cast<int64_t>(wo) * static_cast<int64_t>(sizeof(NbGrad));
}

int gg_mipmap_warp_backward(float* grad_src, float* grad_pyramid, float* grad_grid, void* workspace, const void* grad_out,
                            const void* src, const float* pyramid, const float* grid, int dtype, int64_t N, int C,
                            int hs, int ws, int ho, int wo, int extra_levels, float max_level, float min_level,
                            int padding_mode, void* stream) {
  WarpParams wp;
  int rc = fill_params(&wp, N, C, hs, ws, ho, wo, padding_mode, extra_levels, max_level, min_level);
  if (rc != GG_OK) return rc;
  const int64_t total = N * ho * static_cast<int64_t>(wo);
  if (total == 0) return GG_OK;
  // C == 0 still writes grad_grid (zeros: no channel contributes, and no pixel owes a neighbour a level-of-detail part)
  if ((C > 0 && (!grad_out || !src)) || !grid || (extra_levels > 0 && !pyramid))
    return fail(GG_ERR_BAD_ARG, "mipmap_warp_backward: null tensor");
  if (grad_src && extra_levels > 0 && !grad_pyramid) return fail(GG_ERR_BAD_ARG, "mipmap_warp_backward: grad_src needs grad_pyramid");
  if (!grad_src && !grad_grid) return GG_OK;
  auto st = static_cast<cudaStream_t>(stream);
  const int gridsz = grid_for(total, 256);
  NbGrad* nb = (grad_grid && extra_levels > 0) ? static_cast<NbGrad*>(workspace) : nullptr;
  if (grad_grid && extra_levels > 0 && !nb) return fail(GG_ERR_BAD_ARG, "mipmap_warp_backward: grad_grid needs a workspace");
#define GG_BWD(T_)                                                                                               \
  if (extra_levels > 0)                                                                                          \
    warp_bwd_kernel<T_, true><<<gridsz, 256, 0, st>>>(grad_src, grad_pyramid, grad_grid, nb,                    \
        static_cast<const T_*>(grad_out), static_cast<const T_*>(src), pyramid, grid, wp, total);               \
  else                                                                                                           \
    warp_bwd_kernel<T_, false><<<gridsz, 256, 0, st>>>(grad_src, grad_pyramid, grad_grid, nb,                   \
        static_cast<const T_*>(grad_out), static_cast<const T_*>(src), pyramid, grid, wp, total)
  switch (dtype) {
    case GG_F32: GG_BWD(float); break;
    case GG_F16: GG_BWD(__half); break;
    case GG_BF16: GG_BWD(__nv_bfloat16); break;
    default: return fail(GG_ERR_UNSUPPORTED, "mipmap_warp_backward: dtype %d not supported", dtype);
  }
#undef GG_BWD
  GG_CHECK_LAUNCH("warp_bwd launch");
  if (nb) {
    warp_grid_gather_kernel<<<gridsz, 256, 0, st>>>(grad_grid, nb, ho, wo, total);
    GG_CHECK_LAUNCH("warp_grid_gather launch");
  }
  return GG_OK;
}

}  // extern "C"
