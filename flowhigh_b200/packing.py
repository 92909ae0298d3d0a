"""Host-side weight layout transforms (done once at load time, torch is only the container).

`tapped_conv_weights` turns Conv1d / ConvTranspose1d / Linear weights into the generic
"tapped convolution" form both conv kernels consume:
    out[b, co, P*t + p] = sum_m sum_ci W[p][m][co][ci] * x[b, ci, t + off[p][m]]
`pack_tc` lays W out as the shared-memory image of fh_tc_conv
([p][n_tile][ci_pair][tap][2 chunks][bn rows][8 ci] bf16, K-major no-swizzle core matrices).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np
import torch


@dataclass
class TappedConv:
    w: torch.Tensor            # [P, ntaps, Cout, Cin] fp32
    off: np.ndarray            # [P, ntaps] int32 input-row offsets
    bias: Optional[torch.Tensor]
    P: int
    ntaps: int

    @property
    def cout(self):
        return self.w.shape[2]

    @property
    def cin(self):
        return self.w.shape[3]


def conv1d_taps(weight: torch.Tensor, bias, dilation: int = 1) -> TappedConv:
    """nn.Conv1d(C_in, C_out, k, dilation=d, padding=(k*d-d)//2)  (bigvgan/utils.py:53-54)."""
    cout, cin, k = weight.shape
    w = weight.permute(2, 0, 1).unsqueeze(0).contiguous()  # [1, k, Cout, Cin]
    half = (k * dilation - dilation) // 2
    off = np.array([[j * dilation - half for j in range(k)]], dtype=np.int32)
    return TappedConv(w.float(), off, bias, 1, k)


def linear_taps(weight: torch.Tensor, bias) -> TappedConv:
    cout, cin = weight.shape
    return TappedConv(weight.reshape(1, 1, cout, cin).float().contiguous(), np.zeros((1, 1), np.int32), bias, 1, 1)


def conv_transpose1d_taps(weight: torch.Tensor, bias, stride: int) -> TappedConv:
    """nn.ConvTranspose1d(C_in, C_out, k, stride=u, padding=(k-u)//2) in polyphase form.

    out[u*q + r] = sum_{j = (r+p) mod u + m*u} W[ci, co, j] * x[q + (r + p - j)/u]   (models.py:140-146)
    """
    cin, cout, k = weight.shape
    u = stride
    pad = (k - u) // 2
    ntaps = -(-k // u)
    w = torch.zeros(u, ntaps, cout, cin, dtype=torch.float32, device=weight.device)
    off = np.zeros((u, ntaps), dtype=np.int32)
    for r in range(u):
        j0 = (r + pad) % u
        base = (r + pad - j0) // u
        for m in range(ntaps):
            j = j0 + m * u
            off[r, m] = base - m
            if j < k:
                w[r, m] = weight[:, :, j].t()
    return TappedConv(w, off, bias, u, ntaps)


def split_input(tc: TappedConv, cin_pad: int) -> TappedConv:
    """Weights for a hi + lo split activation operand (precision "fp16x2"): the input channels are doubled,
    [0, cin) multiply the hi halves and [cin_pad, cin_pad + cin) the lo halves, with the SAME weights, so
    W . (hi + lo) is accumulated in fp32 by the ordinary kernel over 2 * cin_pad input channels."""
    P, ntaps, cout, cin = tc.w.shape
    w = torch.zeros(P, ntaps, cout, 2 * cin_pad, dtype=tc.w.dtype, device=tc.w.device)
    w[..., :cin] = tc.w
    w[..., cin_pad:cin_pad + cin] = tc.w
    return TappedConv(w, tc.off, tc.bias, tc.P, tc.ntaps)


def f32_conv_buffers(tc: TappedConv, device):
    """fh_conv1d_taps_f32 operands: w [P][Cout][Cin][ntaps] fp32, off [P][ntaps] int32."""
    w = tc.w.permute(0, 2, 3, 1).contiguous().to(device)
    off = torch.from_numpy(tc.off.copy()).to(device)
    return w, off


def pick_bn(cout_pad: int) -> int:
    # Measured on B200 once the MMA issue loop stopped pacing the kernel (gpurun_out/bd5_*.json): accumulators that fit
    # TMEM twice (2 sub-tiles x bn <= 256 columns) so the epilogue overlaps the next tile beat the wider single-buffered
    # tiles for 192 and 384 output channels (-12 % / -21 %); 768 keeps 3 x 256.
    if cout_pad <= 128:
        return round_up(cout_pad, 16)  # MMA N granularity at M = 128; surplus columns carry zero weights
    if cout_pad <= 256:
        half = cout_pad // 2
        return half if cout_pad % 32 == 0 else round_up(cout_pad, 16)
    if cout_pad % 256 == 0:
        return 256
    for bn in (128, 192, 160, 176, 144, 224, 208, 240):
        if cout_pad % bn == 0:
            return bn
    return 256


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def pack_tc(tc: TappedConv, device, cin_pad: Optional[int] = None, cout_pad: Optional[int] = None,
            bn: Optional[int] = None, dtype=torch.bfloat16, two_cta: bool = False) -> Tuple[torch.Tensor, int, int, int]:
    """-> (packed 16-bit tensor (bf16 or fp16), cin_pad, cout_pad, bn).
    two_cta: layout of the CTA-pair kernel, [P][nt][cp][rank][tap][2][bn/2][8] -- CTA `rank` of a pair fetches the
    bn/2 output channels [rank bn/2, (rank + 1) bn/2) of every weight slot as one contiguous block per ci-pair."""
    P, ntaps, cout, cin = tc.w.shape
    cin_pad = cin_pad or round_up(cin, 8)     # channel counts of the activation buffers: whole 8-channel chunks
    cout_pad = cout_pad or round_up(cout, 8)
    bn = bn or pick_bn(cout_pad)
    n_tiles = -(-cout_pad // bn)
    cin16 = round_up(cin_pad, 16)             # the weight image always carries whole ci-pairs (K = 16 per MMA)
    w = torch.zeros(P, ntaps, n_tiles * bn, cin16, dtype=torch.float32, device=tc.w.device)
    w[:, :, :cout, :cin] = tc.w
    if two_cta:
        # [P][tap][nt][rank][bn/2][cp][2][8] -> [P][nt][cp][rank][tap][2][bn/2][8]
        w = w.reshape(P, ntaps, n_tiles, 2, bn // 2, cin16 // 16, 2, 8).permute(0, 2, 5, 3, 1, 6, 4, 7).contiguous()
        return w.to(dtype).to(device), cin_pad, cout_pad, bn
    # [P][tap][nt][bn][cp][2][8] -> [P][nt][cp][tap][2][bn][8]
    w = w.reshape(P, ntaps, n_tiles, bn, cin16 // 16, 2, 8).permute(0, 2, 4, 1, 5, 3, 6).contiguous()
    return w.to(dtype).to(device), cin_pad, cout_pad, bn


def pad_vec(v: Optional[torch.Tensor], n: int, fill: float = 0.0) -> Optional[torch.Tensor]:
    if v is None:
        return None
    out = torch.full((n,), fill, dtype=torch.float32, device=v.device)
    out[: v.numel()] = v.flatten().float()
    return out
