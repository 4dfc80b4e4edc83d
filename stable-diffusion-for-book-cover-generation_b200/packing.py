"""Host-side weight repacking from diffusers (OIHW / [out,in]) layouts into the kernels' layouts.
Pure torch tensor reshuffles, done once at load time."""
from __future__ import annotations

import torch


def pack_conv3x3(w: torch.Tensor) -> torch.Tensor:
    """(Cout, Cin, 3, 3) -> bf16 [Cout][ky][kx][Cin] flattened to (Cout, 9*Cin): K index = tap*Cin + c."""
    co, ci, kh, kw = w.shape
    return w.permute(0, 2, 3, 1).reshape(co, kh * kw * ci).contiguous().to(torch.bfloat16)


def pack_conv3x3_f32(w: torch.Tensor) -> torch.Tensor:
    co, ci, kh, kw = w.shape
    return w.permute(0, 2, 3, 1).reshape(co, kh * kw * ci).contiguous().float()


def pack_linear(w: torch.Tensor) -> torch.Tensor:
    """(out, in) or (out, in, 1, 1) -> bf16 (out, in)."""
    return w.reshape(w.shape[0], -1).contiguous().to(torch.bfloat16)


def pack_geglu(w: torch.Tensor, b: torch.Tensor, tile: int):
    """GEGLU proj (8C, C): rows [0,4C) = value, [4C,8C) = gate.  Interleave per `tile` columns so each
    output tile of the GEMM holds [tile/2 values | the matching tile/2 gates]."""
    n2 = w.shape[0]
    half = n2 // 2
    h = tile // 2
    assert half % h == 0
    wv, wg = w[:half].reshape(half // h, h, -1), w[half:].reshape(half // h, h, -1)
    bv, bg = b[:half].reshape(half // h, h), b[half:].reshape(half // h, h)
    wp = torch.cat([wv, wg], dim=1).reshape(n2, -1).contiguous().to(torch.bfloat16)
    bp = torch.cat([bv, bg], dim=1).reshape(n2).contiguous().float()
    return wp, bp


def pack_conv_out_tc(w: torch.Tensor, pad_to: int = 32) -> torch.Tensor:
    """conv_out (Cout <= 4, Cin, 3, 3) fp32 -> bf16 [pad_to][9][2*Cin] for the tensor-core path: per tap [hi | lo] with
    hi = bf16(w), lo = bf16(w - hi), so that [x | x] . [hi | lo] restores the fp32 weights to ~2^-17 (the last layer of the network
    feeds the noise prediction directly: plain bf16 weights would cost ~1e-3 of the 1e-2 parity budget).  Rows >= Cout are zero."""
    co, ci, kh, kw = w.shape
    wt = w.permute(0, 2, 3, 1).reshape(co, kh * kw, ci).float()
    hi = wt.to(torch.bfloat16)
    lo = (wt - hi.float()).to(torch.bfloat16)
    out = torch.zeros(pad_to, kh * kw, 2 * ci, dtype=torch.bfloat16, device=w.device)
    out[:co, :, :ci] = hi
    out[:co, :, ci:] = lo
    return out.reshape(pad_to, kh * kw * 2 * ci).contiguous()
