"""CPU restatement of the Spatial Transformer's samplers (test infrastructure -- see oracle/__init__.py).

Follows reference models/spatial_transformers/antialiased_sampling.py:
  Warp.forward :9-16, MipmapWarp.forward :35-60, get_max_coord_distance :62-97, _downsample_2x :111-117,
  _create_stack :119-150, _upsample :155-160, _warp_stack :162-179, _get_coordinates :181-195,
  _get_mipmap_levels :197-210, _sample_mipmap :212-238, BilinearDownsample :241-256.
The third-party arithmetic the reference delegates to PyTorch (F.grid_sample, F.interpolate, F.pad,
F.conv2d; unpinned version, torch 2.11 in this image) is restated here with explicit index arithmetic so
that the integer work (corner indices, reflection, level indices) is spelled out; make_golden.py pins
every function against the reference run on the same inputs.
"""
import math

import torch
import torch.nn.functional as F

PAD_MODES = ("zeros", "border", "reflection")


# ------------------------------------------------------------------------------------ grid_sample (bilinear)
def _reflect(coord, twice_low, twice_high):
    """ATen reflect_coordinates (GridSampler.h): reflect about the pixel-edge interval."""
    if twice_low == twice_high:
        return torch.zeros_like(coord)
    lo = twice_low / 2.0
    span = (twice_high - twice_low) / 2.0
    c = (coord - lo).abs()
    extra = torch.fmod(c, span)
    flips = torch.floor(c / span)
    even = torch.fmod(flips, 2.0) == 0
    return torch.where(even, extra + lo, span - extra + lo)


def source_index(g, size, padding_mode):
    """normalised grid coordinate -> source pixel coordinate, align_corners=False
    (ATen grid_sampler_compute_source_index)."""
    x = ((g + 1.0) * size - 1.0) / 2.0
    if padding_mode == "border":
        x = _clip(x, size)
    elif padding_mode == "reflection":
        x = _clip(_reflect(x, -1, 2 * size - 1), size)
    return x


def _clip(x, size):
    """ATen clip_coordinates(_set_grad): clamp to [0, size-1]; the gradient is zero AT and beyond the borders
    (torch.clamp would pass it at the border itself)."""
    inside = (x > 0) & (x < size - 1)
    return torch.where(inside, x, x.detach().clamp(0, size - 1))


def grid_sample_bilinear(img, grid, padding_mode="border"):
    """F.grid_sample(img, grid, mode='bilinear', padding_mode, align_corners=False) restated.
    Returns (out, corner indices (x0, y0)) -- the integer corner indices are exposed for exact checks."""
    assert padding_mode in PAD_MODES
    n, c, h, w = img.shape
    ix = source_index(grid[..., 0], w, padding_mode)
    iy = source_index(grid[..., 1], h, padding_mode)
    x0, y0 = torch.floor(ix), torch.floor(iy)
    x1, y1 = x0 + 1, y0 + 1
    w_nw = (x1 - ix) * (y1 - iy)
    w_ne = (ix - x0) * (y1 - iy)
    w_sw = (x1 - ix) * (iy - y0)
    w_se = (ix - x0) * (iy - y0)
    flat = img.reshape(n, c, h * w)

    def tap(xc, yc, wt):
        ok = (xc >= 0) & (xc <= w - 1) & (yc >= 0) & (yc <= h - 1)
        idx = (yc.clamp(0, h - 1) * w + xc.clamp(0, w - 1)).long().reshape(n, 1, -1).expand(n, c, -1)
        val = torch.gather(flat, 2, idx).reshape(n, c, *xc.shape[1:])
        return val * (wt * ok).unsqueeze(1)

    out = tap(x0, y0, w_nw) + tap(x1, y0, w_ne) + tap(x0, y1, w_sw) + tap(x1, y1, w_se)
    return out, (x0.long(), y0.long())


def warp_ref(img, grid, padding_mode="border"):
    """Warp.forward (antialiased_sampling.py:15-16)."""
    return grid_sample_bilinear(img, grid, padding_mode)[0]


# ------------------------------------------------------------------------------------ mip pyramid pieces
def blur_filter():
    f = torch.tensor([1.0, 3.0, 3.0, 1.0])
    f = f[:, None] * f[None, :]
    return f / f.sum()


def downsample_2x(x):
    """_downsample_2x (:111-117): ReflectionPad2d(1) then depthwise [1,3,3,1]^2/64, stride 2."""
    c = x.shape[1]
    x = F.pad(x, (1, 1, 1, 1), mode="reflect")
    return F.conv2d(x, blur_filter().to(x.dtype)[None, None].repeat(c, 1, 1, 1), stride=2, groups=c)


def upsample_bilinear(x, factor):
    """_upsample (:155-160) = F.interpolate(scale_factor=factor, bilinear, align_corners=False), restated:
    src = (dst + 0.5)/factor - 0.5 clamped at 0; i1 = min(i0 + 1, size - 1)."""
    n, c, h, w = x.shape
    factor = int(factor)

    def axis(size):
        dst = torch.arange(size * factor, dtype=x.dtype)
        src = ((dst + 0.5) * (1.0 / factor) - 0.5).clamp(min=0)
        i0 = src.floor().long()
        i1 = torch.where(i0 < size - 1, i0 + 1, i0)
        lam = src - i0
        return i0, i1, lam

    y0, y1, ly = axis(h)
    x0, x1, lx = axis(w)
    top = x[:, :, y0][:, :, :, x0] * (1 - lx) + x[:, :, y0][:, :, :, x1] * lx
    bot = x[:, :, y1][:, :, :, x0] * (1 - lx) + x[:, :, y1][:, :, :, x1] * lx
    return top * (1 - ly)[:, None] + bot * ly[:, None]


def pow2_padding(width):
    """_create_stack (:130-137): pad a non power-of-two (square) source up to the next power of two."""
    log_size = math.log2(width)
    if float(log_size).is_integer():
        return 0, 0
    target = 2 ** math.ceil(log_size)
    total = target - width
    left = int(total // 2)
    return left, int(total - left)


def create_stack(x, num_levels):
    """_create_stack (:119-150): level i = upsample_{2^i}(downsample_2x^i(x)); D = num_levels."""
    left, right = pow2_padding(x.shape[-1])
    if left or right:
        x = F.pad(x, (left, right, left, right), mode="reflect")
    levels = [x]
    cur = x
    for i in range(1, num_levels):
        cur = downsample_2x(cur)
        levels.append(upsample_bilinear(cur, 2 ** i))
    stack = torch.stack(levels, dim=2)
    if left or right:
        stack = stack[:, :, :, left:-right, left:-right]
    return stack


# ------------------------------------------------------------------------------------ level of detail
def lod_coordinates(grid, height, width):
    """_get_coordinates (:181-195) -- note the (size-1) scaling, unlike the sampler's align_corners=False."""
    x = (width - 1.0) * (grid[..., 0] + 1.0) / 2.0
    y = (height - 1.0) * (grid[..., 1] + 1.0) / 2.0
    return torch.stack([x, y], dim=3)


def max_coord_distance(coords):
    """get_max_coord_distance (:62-97): replicate-padded 4-neighbour distances, clamped at 1, max."""
    p = F.pad(coords.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="replicate").permute(0, 2, 3, 1)
    neigh = [p[:, 1:-1, :-2], p[:, 1:-1, 2:], p[:, :-2, 1:-1], p[:, 2:, 1:-1]]  # left, right, up, down
    dists = [((o - coords) ** 2).sum(dim=3).clamp(min=1.0) ** 0.5 for o in neigh]
    return torch.stack(dists).max(dim=0).values


def mipmap_levels(grid, height, width, max_num_levels, min_level=0.0):
    """_get_mipmap_levels (:197-210) + the min_level clamp of forward (:49)."""
    d = max_coord_distance(lod_coordinates(grid, height, width))
    return torch.log2(d).clamp(min=0.0, max=max_num_levels - 1.0).clamp(min=min_level)


def mipmap_warp_ref(x, grid, max_num_levels=8, min_level=0.0, padding_mode="border", return_aux=False):
    """MipmapWarp.forward (:35-60).  Returns out [, dict(levels, level_0, level_1, num_levels, levels_map)]."""
    n, c, h, w = x.shape
    levels = mipmap_levels(grid, h, w, max_num_levels, min_level)
    num_levels = int(levels.max().ceil().item()) + 1                      # :52 (batch-global, host sync)
    stack = create_stack(x, num_levels)                                   # (N, C, D, H, W)
    d = stack.shape[2]
    warped = grid_sample_bilinear(stack.reshape(n, c * d, h, w), grid, padding_mode)[0]
    warped = warped.reshape(n, c, d, *grid.shape[1:3])
    l0 = levels.floor().long()                                            # :228-229
    l1 = levels.ceil().long()
    idx0 = l0[:, None, None].expand(n, c, 1, *l0.shape[1:])
    idx1 = l1[:, None, None].expand(n, c, 1, *l1.shape[1:])
    o0 = torch.gather(warped, 2, idx0)[:, :, 0]
    o1 = torch.gather(warped, 2, idx1)[:, :, 0]
    out = o0 + (levels % 1.0)[:, None] * (o1 - o0)                        # :235-236
    if return_aux:
        return out, {"levels": levels, "level_0": l0, "level_1": l1, "num_levels": num_levels,
                     "levels_map": levels / (max_num_levels - 1.0)}
    return out


# ------------------------------------------------------------------------------------ where the gradient is decided
# The sampler's gradient is piecewise smooth.  It jumps where a source coordinate crosses an integer (the bilinear
# corners change), a clip bound or a reflection fold, where the level crosses an integer or a clamp, and where the
# arg-max neighbour of the level of detail changes.  Near such a point, the last bits of an fp32 evaluation decide
# which side is taken, so an fp32 kernel and a float64 oracle may both be right and still differ by O(1).  These
# helpers mark the pixels where no such point is within a tolerance, measured on the oracle's own coordinates.
def coordinate_decided(g, size, padding_mode, tol=1e-3):
    """bool, per grid value `g` along an axis of `size` source pixels: the source coordinate is more than `tol` px from
    an integer, from the clip bounds 0 and size-1 (border, reflection) and from the folds -1/2 and size-1/2
    (reflection).  A coordinate clamped to a bound from more than `tol` px beyond it is decided: both sides agree."""
    raw = ((g + 1.0) * size - 1.0) / 2.0
    ok = torch.ones_like(raw, dtype=torch.bool)
    pre = raw
    if padding_mode == "reflection":
        pre = _reflect(raw, -1, 2 * size - 1)
        ok &= ((pre + 0.5).abs() > tol) & ((pre - (size - 0.5)).abs() > tol)
    clamped = torch.zeros_like(ok)
    if padding_mode != "zeros":
        ok &= (pre.abs() > tol) & ((pre - (size - 1)).abs() > tol)
        clamped = (pre < 0) | (pre > size - 1)
    post = source_index(g, size, padding_mode)
    return ok & (clamped | ((post - post.round()).abs() > tol))


def level_decided(grid, height, width, max_num_levels, min_level=0.0, tol=1e-4, axis_ties=False):
    """bool (N, Ho, Wo): the level of detail and the neighbour its gradient goes to are decided.
    - the arg-max squared neighbour distance is not within `tol` of 1 (the clamp(min=1) edge);
    - the unclamped level is more than `tol` from max_level and min_level, and, where it is not clamped, from an integer;
    - where the level gradient flows, the largest clamped distance beats the runner-up by more than `tol` relative.
      With `axis_ties`, a tie between left and right only, or up and down only, is allowed: on an affine grid those two
      distances are the same function of the grid, so a reduction such as d loss / d theta does not depend on the winner
      (a per-pixel gradient does: the part owed to the winner goes to a different pixel)."""
    max_level = max_num_levels - 1.0
    c = lod_coordinates(grid, height, width)
    p = F.pad(c.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="replicate").permute(0, 2, 3, 1)
    neigh = [p[:, 1:-1, :-2], p[:, 1:-1, 2:], p[:, :-2, 1:-1], p[:, 2:, 1:-1]]  # left, right, up, down
    sq = torch.stack([((o - c) ** 2).sum(dim=3) for o in neigh])
    m = sq.max(dim=0).values
    all_clamped = m < 1.0 - tol
    raw = 0.5 * torch.log2(m.clamp(min=1.0))
    ok = (m - 1.0).abs() > tol
    ok &= all_clamped | (((raw - max_level).abs() > tol) & ((raw - min_level).abs() > tol))
    flows = (~all_clamped) & (raw < max_level) & (raw > min_level)
    ok &= ~flows | ((raw - raw.round()).abs() > tol)
    top = sq.clamp(min=1.0).sqrt().topk(3, dim=0)
    d, k = top.values, top.indices
    clear = (d[0] - d[1]) > tol * d[0]
    if axis_ties:
        pair = torch.minimum(k[0], k[1]) * 4 + torch.maximum(k[0], k[1])
        axis_pair = (pair == 1) | (pair == 11)                      # {left, right} or {up, down}
        clear |= axis_pair & ((d[1] - d[2]) > tol * d[0])
    return ok & (~flows | clear)


def decided_pixels(grid, height, width, padding_mode="border", max_num_levels=None, min_level=0.0, coord_tol=1e-3,
                   level_tol=1e-4, axis_ties=False):
    """bool (N, Ho, Wo): pixels whose grid gradient is a smooth function of the grid near `grid`, for a source of
    height x width.  The pixel's own source coordinates must be decided (coordinate_decided).  With mip levels
    (max_num_levels not None), so must the level of detail (level_decided) of the pixel and of its four neighbours: a
    pixel's grid gradient collects the level-of-detail parts its neighbours owe it, and their sampled values enter those
    parts, but not their sampling derivatives."""
    ok = coordinate_decided(grid[..., 0], width, padding_mode, coord_tol) & \
        coordinate_decided(grid[..., 1], height, padding_mode, coord_tol)
    if max_num_levels is None:
        return ok
    lod = level_decided(grid, height, width, max_num_levels, min_level, level_tol, axis_ties)
    q = F.pad(lod[:, None].double(), (1, 1, 1, 1), mode="replicate")[:, 0] > 0.5
    return ok & lod & q[:, 1:-1, :-2] & q[:, 1:-1, 2:] & q[:, :-2, 1:-1] & q[:, 2:, 1:-1]


# ------------------------------------------------------------------------------------ BilinearDownsample
def bilinear_downsample_ref(x, stride):
    """BilinearDownsample.forward (:241-256): reflect-pad stride//2, separable tent filter, stride s."""
    c = x.shape[1]
    ramp = torch.arange(1, 2 * stride + 1, 2, dtype=torch.float64)
    tent = torch.cat([ramp, ramp.flip(0)])
    tent = (tent / tent.sum()).to(x.dtype)
    x = F.pad(x, [int(stride / 2)] * 4, mode="reflect")
    x = F.conv2d(x, tent.reshape(1, 1, 1, -1).repeat(c, 1, 1, 1), stride=(1, stride), groups=c)
    return F.conv2d(x, tent.reshape(1, 1, -1, 1).repeat(c, 1, 1, 1), stride=(stride, 1), groups=c)


def affine_grid_ref(theta, size):
    """F.affine_grid(theta, size, align_corners=False) restated: base coords (2i + 1)/S - 1, times theta^T."""
    n, _, h, w = size
    xs = (2 * torch.arange(w, dtype=theta.dtype) + 1) / w - 1
    ys = (2 * torch.arange(h, dtype=theta.dtype) + 1) / h - 1
    base = torch.stack([xs[None, :].expand(h, w), ys[:, None].expand(h, w), torch.ones(h, w, dtype=theta.dtype)], dim=2)
    return torch.einsum("hwk,njk->nhwj", base, theta)
