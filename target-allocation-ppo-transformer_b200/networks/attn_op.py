"""Fused self-attention over the 5-token window for the PPO update (csrc/ppo_attn.cu), as an autograd function.

attention5(q, k, v, pad_mask): q [n, nq, 128] (nq = 5 or 1), k, v [n, 5, 128] (arbitrary row stride: views into the packed
in_proj output), pad_mask [n, 5] bool -> [n, nq, 128].  8 heads of 16, scores / sqrt(16), -inf on padded keys, softmax,
weighted sum - what nn.MultiheadAttention computes inside the reference's encoder layers (transformer_net.py:34-43,63).
CUDA fp32 only; the network falls back to plain tensor ops elsewhere (CPU tests, autocast)."""
import ctypes as C

import torch

from .. import _capi


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _rows(t):
    """Row stride (floats) of a [n, s, 128] tensor whose rows are contiguous and evenly spaced."""
    n, s, d = t.shape
    if t.stride(2) != 1 or (n > 1 and t.stride(0) != s * t.stride(1)):
        return None
    return t.stride(1)


class _Attention5(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, pad_u8):
        n, nq, _ = q.shape
        out = torch.empty(n, nq, 128, dtype=torch.float32, device=q.device)
        lib = _capi.load()
        stream = C.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)
        _capi.check(lib.ppo_attn5_forward(_ptr(q), _rows(q), _ptr(k), _ptr(v), _rows(k), _ptr(pad_u8), n, nq, _ptr(out),
                                          q.device.index, stream))
        ctx.save_for_backward(q, k, v, pad_u8)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        q, k, v, pad_u8 = ctx.saved_tensors
        n, nq, _ = q.shape
        grad_out = grad_out.contiguous()
        # gradients are produced with the strides of their inputs, so views into a packed buffer stay views
        gq, gk, gv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        if _rows(gq) != _rows(q) or _rows(gk) != _rows(k) or _rows(gv) != _rows(k):
            gq, gk, gv = (torch.empty_strided(t.shape, t.stride(), dtype=t.dtype, device=t.device) for t in (q, k, v))
        lib = _capi.load()
        stream = C.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)
        _capi.check(lib.ppo_attn5_backward(_ptr(q), _rows(q), _ptr(k), _ptr(v), _rows(k), _ptr(pad_u8), n, nq,
                                           _ptr(grad_out), _ptr(gq), _ptr(gk), _ptr(gv), q.device.index, stream))
        return gq, gk, gv, None


def usable(q, k, v):
    return (q.is_cuda and q.dtype == k.dtype == v.dtype == torch.float32 and not torch.is_autocast_enabled()
            and q.shape[-1] == 128 and k.shape[1] == 5 and q.shape[1] in (1, 5)
            and _rows(q) is not None and _rows(k) is not None and _rows(k) == _rows(v)
            and _rows(q) % 4 == 0 and _rows(k) % 4 == 0 and q.data_ptr() % 16 == 0 and k.data_ptr() % 16 == 0
            and v.data_ptr() % 16 == 0)


def attention5(q, k, v, pad_mask):
    return _Attention5.apply(q, k, v, pad_mask.to(torch.uint8).contiguous())
