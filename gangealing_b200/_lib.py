"""ctypes binding of libgg_b200.so -- the only door between Python and the sm_100a kernels.

PyTorch is used for device memory and streams only: every op allocates its outputs with torch,
hands raw device pointers + the current CUDA stream to the C ABI (include/gg_b200.h) and raises
RuntimeError with gg_last_error() on a non-zero return.  If the shared object is missing the import
of any op fails loudly (no fallback path exists).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgg_b200.so")

GG_F32, GG_F16, GG_BF16 = 0, 1, 2
PAD_MODES = {"zeros": 0, "border": 1, "reflection": 2}

_c = ctypes
_P, _I, _L, _F = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float

# name -> (restype, argtypes); must list every symbol declared in include/gg_b200.h
SIGNATURES = {
    "gg_version": (_I, []),
    "gg_last_error": (_c.c_char_p, []),
    "gg_sm_count": (_I, []),
    "gg_fused_bias_act": (_I, [_P, _P, _P, _P, _I, _I, _I, _F, _F, _L, _L, _L, _P]),
    "gg_noise_bias_act": (_I, [_P, _P, _P, _P, _P, _P, _I, _F, _F, _L, _L, _L, _P]),
    "gg_channel_scale_workspace": (_L, [_L, _L]),
    "gg_channel_scale": (_I, [_P, _P, _P, _P, _P, _P, _I, _L, _L, _P]),
    "gg_bias_act_backward_workspace": (_L, [_L, _L, _L]),
    "gg_bias_act_backward": (_I, [_P, _P, _P, _P, _P, _I, _F, _F, _L, _L, _L, _P]),
    "gg_upfirdn2d": (_I, [_P, _P, _P, _I, _L] + [_I] * 12 + [_P]),
    "gg_blur_noise_bias_act": (_I, [_P] * 7 + [_I, _L, _L] + [_I] * 9 + [_F, _F, _P]),
    "gg_mipmap_pyramid_elems": (_L, [_L, _I, _I, _I]),
    "gg_mipmap_build": (_I, [_P, _P, _I, _L, _I, _I, _I, _P]),
    "gg_mipmap_build_backward": (_I, [_P, _P, _L, _I, _I, _I, _P]),
    "gg_mipmap_warp_forward": (_I, [_P] * 5 + [_I, _L] + [_I] * 6 + [_F, _F, _I, _P]),
    "gg_warp_sample_indices": (_I, [_P, _P, _L, _I, _I, _I, _I, _F, _F, _I, _P]),
    "gg_stn_sample_forward": (_I, [_P] * 11 + [_I, _I, _L] + [_I] * 9 + [_F, _F, _I, _P]),
    "gg_modconv_wsq": (_I, [_P, _P, _I, _I, _I, _P]),
    "gg_modconv_demod": (_I, [_P, _P, _P, _F, _F, _I, _I, _I, _P]),
    "gg_modconv_demod_batched": (_I, [_I, _P, _P, _P, _P, _P, _P, _F, _I, _P]),
    "gg_modconv_modulate": (_I, [_P, _P, _P, _P, _F, _I, _I, _I, _I, _I, _P]),
    "gg_noise_bias_act_nhwc": (_I, [_P] * 6 + [_I, _F, _F, _L, _I, _L, _P]),
    "gg_nhwc_rowwise_workspace": (_L, [_L, _I, _L]),
    "gg_channel_scale_nhwc": (_I, [_P] * 6 + [_I, _L, _I, _L, _P]),
    "gg_bias_act_backward_nhwc": (_I, [_P] * 5 + [_I, _F, _F, _L, _I, _L, _P]),
    "gg_blur_nhwc_workspace": (_L, [_I, _L] + [_I] * 9),
    "gg_blur_nhwc": (_I, [_P] * 12 + [_I, _L] + [_I] * 12 + [_F, _F, _P]),
    "gg_styled_tail_nhwc": (_I, [_P] * 12 + [_I, _I, _F, _F, _L, _I, _L, _P]),
    "gg_styled_tail_backward_workspace": (_L, [_I, _L, _I, _L]),
    "gg_styled_tail_backward_nhwc": (_I, [_P] * 12 + [_I, _F, _F, _L, _I, _L, _L, _P]),
    "gg_tent_downsample_forward": (_I, [_P] * 4 + [_L, _I, _I, _I, _I, _P]),
    "gg_tent_downsample_backward": (_I, [_P] * 4 + [_L, _I, _I, _I, _I, _P]),
    "gg_feature_distance_workspace": (_L, [_L, _I, _L]),
    "gg_feature_distance_forward": (_I, [_P] * 5 + [_I, _L, _I, _L, _F, _P]),
    "gg_feature_distance_backward": (_I, [_P] * 6 + [_I, _L, _I, _L, _F, _P]),
    "gg_bias_relu_pool_nhwc_forward": (_I, [_P, _P, _P, _P, _I, _L, _I, _I, _I, _P]),
    "gg_bias_relu_pool_nhwc_backward": (_I, [_P, _P, _P, _P, _I, _L, _I, _I, _I, _P]),
    "gg_to_rgb_nhwc_workspace": (_L, [_L, _I, _L]),
    "gg_to_rgb_nhwc_forward": (_I, [_P] * 5 + [_L, _I, _L, _P]),
    "gg_to_rgb_nhwc_backward": (_I, [_P] * 6 + [_L, _I, _L, _P]),
    "gg_nn_argmin_workspace": (_L, [_L, _L]),
    "gg_nn_argmin": (_I, [_P, _P, _P, _P, _L, _L, _I, _P]),
    "gg_splat2d_lookup_forward": (_I, [_P] * 8 + [_L, _L, _I, _I, _I, _I, _I, _F, _F, _I, _P]),
    "gg_scale_cast_multi": (_I, [_P, _P, _P, _I, _I, _P]),
    "gg_adam_ema_step": (_I, [_P, _P, _P, _I, _I, _P, _c.c_double, _c.c_double, _c.c_double, _c.c_double, _P]),
    "gg_tv_loss_workspace": (_L, [_L, _I, _I]),
    "gg_tv_loss_forward": (_I, [_P, _P, _P, _L, _I, _I, _P]),
    "gg_tv_loss_backward": (_I, [_P, _P, _P, _L, _I, _I, _P]),
    "gg_splat2d_workspace": (_L, [_L, _I, _I, _I]),
    "gg_splat2d_forward": (_I, [_P] * 6 + [_L, _L, _I, _I, _I, _I, _P]),
    "gg_flow_compose_forward": (_I, [_P] * 7 + [_L, _I, _I, _I, _P]),
    "gg_flow_compose_backward_workspace": (_L, [_L, _I, _I, _I]),
    "gg_flow_compose_backward": (_I, [_P] * 11 + [_L, _I, _I, _I, _P]),
    "gg_mipmap_warp_backward_workspace": (_L, [_L, _I, _I]),
    "gg_mipmap_warp_backward": (_I, [_P] * 8 + [_I, _L] + [_I] * 6 + [_F, _F, _I, _P]),
}

_dll = None
CALLS = 0  # C-ABI calls that launched device work (bench.py reports the count as gpu_launches; >= 1 kernel each)


def load():
    """Load (once) and type the shared library.  Raises RuntimeError if it has not been built."""
    global _dll
    if _dll is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libgg_b200.so is missing (%s): build it with `python -m gangealing_b200.build` "
                "(there is no CPU/PyTorch fallback for these ops)" % LIB_PATH)
        dll = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(dll, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _dll = dll
    return _dll


def check(rc, what):
    global CALLS
    CALLS += 1
    if rc != 0:
        msg = load().gg_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))


def dtype_code(t):
    d = t.dtype
    if d == torch.float32:
        return GG_F32
    if d == torch.float16:
        return GG_F16
    if d == torch.bfloat16:
        return GG_BF16
    raise RuntimeError("gangealing_b200: dtype %s is not supported (float32/float16/bfloat16)" % d)


def require_cuda(*tensors):
    """Mirror of the reference's CHECK_CUDA (models/stylegan2/op/upfirdn2d.cpp:8): CUDA tensors only."""
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("gangealing_b200 ops run on CUDA tensors only (got a %s tensor); "
                               "the CPU restatement lives in oracle/ and is test infrastructure" % t.device.type)
        if t.device.index != torch.cuda.current_device():
            # the C ABI launches on the CURRENT device's stream (one process per GPU, like the reference's torchrun
            # recipe): refuse a tensor of another device instead of launching on the wrong one
            raise RuntimeError("gangealing_b200: tensor lives on %s but the current device is cuda:%d; wrap the call in "
                               "`with torch.cuda.device(tensor.device):`" % (t.device, torch.cuda.current_device()))


def ptr(t):
    return None if t is None else t.data_ptr()


def is_nhwc(t):
    """True for a 4-D fp32 / bf16 tensor stored channels-last (and not also plain-contiguous).  The channels-last kernel
    family moves 16 bytes of channels at a time: callers additionally check C % nhwc_vec(t) (or the blur's multiple)."""
    return (t.dim() == 4 and t.dtype in (torch.float32, torch.bfloat16) and t.shape[1] > 1 and t.shape[2] * t.shape[3] > 1
            and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous())


def nhwc_vec(t):
    """Channels per 16-byte access of the channels-last kernels: 4 (fp32) or 8 (bf16)."""
    return 8 if t.dtype == torch.bfloat16 else 4


def tensor_cache(t):
    """Per-tensor-object memo, invalidated when the tensor is modified in place.  (Keyed on the Python object, not on
    data_ptr: a freed temporary's address can be handed to a different tensor.)"""
    # the stamp also carries the storage address, device and dtype: `.data` writes (the reference's own
    # accumulate(), weight surgery) and module.to(device) keep the Python object and its version counter
    stamp = (t._version, t.data_ptr(), t.device, t.dtype)
    ent = getattr(t, "_gg_cache", None)
    if ent is None or ent[0] != stamp:
        ent = (stamp, {})
        try:
            t._gg_cache = ent
        except Exception:
            pass
    return ent[1]


def filter_is_separable(kernel):
    """Rank-1 test of a (<=4x4) FIR filter, memoised on the tensor object: one host read per distinct filter."""
    memo = tensor_cache(kernel)
    v = memo.get("separable")
    if v is None:
        k = kernel.detach().float().cpu()
        big = k.abs().max()
        if big == 0:
            v = True
        else:
            i0, j0 = divmod(int(k.abs().argmax()), k.shape[1])
            v = bool((k - torch.outer(k[:, j0], k[i0, :]) / k[i0, j0]).abs().max() <= 1e-6 * big)
        memo["separable"] = v
    return v


def flipped_filter(kernel):
    """flip(kernel, [0, 1]) (the adjoint resampler's taps), memoised on the filter object so that repeated backward
    passes neither re-launch the flip nor re-test separability (a host read: illegal during graph capture)."""
    memo = tensor_cache(kernel)
    f = memo.get("flipped")
    if f is None:
        f = torch.flip(kernel.detach(), [0, 1])
        fm = tensor_cache(f)
        fm["flipped"] = kernel.detach()
        if "separable" in memo:
            fm["separable"] = memo["separable"]
        memo["flipped"] = f
    return f


def invalidate(t):
    """Drop the memo of a tensor that was rewritten through `.data` IN PLACE at the same address (which no stamp can see):
    call it from weight-loading / conversion hooks."""
    try:
        t._gg_cache = None
    except Exception:
        pass


def workspace(nbytes, device):
    """A device scratch buffer of at least `nbytes` bytes from PyTorch's caching allocator (which aligns blocks to 512 B)."""
    return torch.empty(max(1, (int(nbytes) + 3) // 4), dtype=torch.float32, device=device)


def stream():
    return torch.cuda.current_stream().cuda_stream


def sm_count():
    return load().gg_sm_count()


def ship_table(slot, payload):
    """Copy a small CPU tensor `payload` into the pinned buffer slot["host"] and on to slot["dev"] (async, current stream).
    The pinned buffer is reused every step, and in an eager loop the host may run a whole step ahead of the GPU: before it
    is overwritten, wait for the previous copy OUT of it (an event recorded right after that copy).  Inside a CUDA-graph
    capture no event is recorded or waited on (the table is shipped once per capture; replays re-read the pinned buffer,
    which nothing rewrites while pointers stay put)."""
    capturing = torch.cuda.is_current_stream_capturing()
    ev = slot.get("event")
    if ev is not None and not capturing:   # event waits are illegal while a (global-mode) capture is open; torch.cuda.graph
        ev.synchronize()                   # synchronises the device before it starts capturing, so nothing is in flight then
    slot["host"].copy_(payload)
    slot["dev"].copy_(slot["host"], non_blocking=True)
    if capturing:
        slot["event"] = None
    else:
        ev = torch.cuda.Event()
        ev.record()
        slot["event"] = ev

