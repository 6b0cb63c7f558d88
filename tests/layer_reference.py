"""fp64 references of single generator layers, each fed one layer's own input.

TEST INFRASTRUCTURE ONLY: nothing under ``lip2speech-unit_b200/`` imports this file.

The CPU oracle (``oracle/vocoder_oracle.py``) runs the whole stack, so comparing it with the device waveform mixes the
rounding of every layer.  The functions here run ONE layer in fp64 on the input the device actually produced for it (a
debug tap of the previous layer), so errors do not compound and a per-element tolerance can sit far below the
end-to-end noise.  Every tensor is channels-last (B, L, C), like the taps, and every function works on whichever
device its inputs live on.

Operand rounding follows what the kernels store (``mode``):
  None / "fp32"  no rounding (the fp32 mode keeps fp32 operands; the reference carries them in fp64)
  "bf16"         conv weights bf16(w) of the fp32 folded weights (round to nearest even, as l2s_finalize); every
                 conv input activation as the tensor-core epilogues write it: v = bf16(x), lrelu on the bf16 value with
                 slope bf16(0.1), result rounded to bf16 (conv_common.cuh, lrelu_bf16x2)
  "bf16_simt"    the CUDA-core bf16 convs (knob force_simt): bf16 weights, activation bf16(lrelu(x)) of the fp32 value
  "tf32"         conv weights and conv input activations rounded to nearest (ties away from zero) tf32, as
                 l2s_finalize and the tf32 epilogues do (cvt.rna.tf32.f32)
Biases, the residual stream, branch sums and the waveform head stay unrounded in every mode.
"""
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle import vocoder_oracle as vo

LRELU_SLOPE = vo.LRELU_SLOPE


# --------------------------------------------------------------------------- rounding

def bf16(x: torch.Tensor) -> torch.Tensor:
    """Round to bf16 the way the device does it: from the fp32 value, to nearest even."""
    return x.float().to(torch.bfloat16).to(x.dtype if x.is_floating_point() else torch.float64)


def tf32_rna(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> tf32 (10 mantissa bits), round to nearest, ties away from zero (cvt.rna.tf32.f32)."""
    u = x.float().contiguous().view(torch.int32)
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32).to(x.dtype)


def tf32_trunc(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> tf32 by dropping the low 13 mantissa bits (round toward zero)."""
    u = x.float().contiguous().view(torch.int32)
    return (u & ~0x1FFF).view(torch.float32).to(x.dtype)


def round_weight(w: torch.Tensor, mode: Optional[str]) -> torch.Tensor:
    if mode in ("bf16", "bf16_simt"):
        return bf16(w)
    if mode == "tf32":
        return tf32_rna(w)
    return w


def activate(x: torch.Tensor, mode: Optional[str], slope: float = LRELU_SLOPE) -> torch.Tensor:
    """A conv's input operand: leaky_relu(x) as the producing epilogue stores it, returned in fp64."""
    if mode == "bf16":
        v = x.float().to(torch.bfloat16)
        s = torch.tensor(slope, dtype=torch.float32).to(torch.bfloat16)
        return torch.maximum(v, v * s).double()          # bf16 * bf16 -> product rounded to bf16, like HMUL2
    if mode == "bf16_simt":
        v = x.float()
        return bf16(torch.where(v > 0, v, v * slope)).double()
    if mode == "tf32":
        v = x.float()
        return tf32_rna(torch.maximum(v, v * slope)).double()
    return F.leaky_relu(x.double(), slope)


def layer_weights(sd: Dict[str, torch.Tensor], mode: Optional[str]) -> Dict[str, torch.Tensor]:
    """fp64 weights as the device holds them: folded in fp32 as remove_weight_norm() does, conv weights rounded per
    ``mode`` (conv_post and the front end are fp32 in every mode)."""
    w = vo.fold_weight_norm(sd)
    out = {}
    for k, v in w.items():
        conv = k.endswith(".weight") and (k.startswith(("conv_pre.", "ups.", "resblocks.")))
        out[k] = (round_weight(v, mode) if conv else v).double()
    return out


def to_device(w: Dict[str, torch.Tensor], device) -> Dict[str, torch.Tensor]:
    return {k: v.to(device) for k, v in w.items()}


# --------------------------------------------------------------------------- layers

def front_end(sd: Dict[str, torch.Tensor], h, code, mel=None, spkr=None, unit_only: bool = False) -> torch.Tensor:
    """The oracle's conditioning tensor ``cond`` (B, T, model_in_dim) in fp64, from the test's own inputs."""
    taps = {}
    folded = vo.fold_weight_norm(sd)
    if unit_only:
        vo.code_generator_forward(folded, h, code, spkr, taps=taps)
    else:
        vo.mel_code_generator_forward(folded, h, code, mel, spkr, taps=taps)
    return taps["cond"].transpose(1, 2).contiguous()


def _conv(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, **kw) -> torch.Tensor:
    return F.conv1d(x.transpose(1, 2), w, b, **kw).transpose(1, 2).contiguous()


def conv_pre(w, cond: torch.Tensor) -> torch.Tensor:
    """conv_pre (k = 7) on the cond operand; returns the raw output (the device keeps only leaky_relu(0.1) of it)."""
    return _conv(cond.double(), w["conv_pre.weight"], w["conv_pre.bias"], padding=3)


def upsample(w, h, i: int, a: torch.Tensor) -> torch.Tensor:
    """ups[i] (ConvTranspose1d, stride u, padding (k - u) // 2) on its activated operand ``a``."""
    u, k = h["upsample_rates"][i], h["upsample_kernel_sizes"][i]
    y = F.conv_transpose1d(a.double().transpose(1, 2), w[f"ups.{i}.weight"], w[f"ups.{i}.bias"], stride=u,
                           padding=(k - u) // 2)
    return y.transpose(1, 2).contiguous()


def mrf(w, h, i: int, x: torch.Tensor, mode: Optional[str]) -> torch.Tensor:
    """MRF stage i: every ResBlock1 of the stage on the upsampler output ``x`` (fp32 raw), then the mean over
    branches.  Only conv operands are rounded (per ``mode``); the residual stream and the branch sum stay fp64."""
    nk = len(h["resblock_kernel_sizes"])
    x = x.double()
    total = None
    for j, (rk, dil) in enumerate(zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"])):
        n = i * nk + j
        y = x
        for m, d in enumerate(dil):
            t = _conv(activate(y, mode), w[f"resblocks.{n}.convs1.{m}.weight"], w[f"resblocks.{n}.convs1.{m}.bias"],
                      dilation=d, padding=vo.get_padding(rk, d))
            t = _conv(activate(t, mode), w[f"resblocks.{n}.convs2.{m}.weight"], w[f"resblocks.{n}.convs2.{m}.bias"],
                      padding=vo.get_padding(rk, 1))
            y = y + t
        total = y if total is None else total + y
    return total / nk


def head(w, x: torch.Tensor) -> torch.Tensor:
    """leaky_relu(0.01), conv_post (k = 7, fp32 weights in every mode), tanh: (B, L) waveform from the last MRF output."""
    y = _conv(F.leaky_relu(x.double(), 0.01), w["conv_post.weight"], w["conv_post.bias"], padding=3)
    return torch.tanh(y[..., 0])
