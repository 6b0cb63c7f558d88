"""CPU checks behind tests/test_gpu_layer_parity.py, and of the channel counts l2s_create accepts.

1. The layer references of tests/layer_reference.py, with rounding off and chained on their own outputs, must
   reproduce the oracle's taps (conv_pre, ups.i, mrf.i) and waveform in fp64 up to summation order.  A wrong
   decomposition (a missing activation, a wrong padding, the branch mean taken wrongly) would otherwise make every
   per-layer GPU comparison meaningless.
2. The rounding helpers match the device conventions they claim (bf16 round to nearest even, tf32 round to nearest
   ties away / truncation, the bf16 leaky-ReLU of the tensor-core epilogues).
3. Every conv except conv_pre reads its input with a row pitch of cin_pad (cin padded to a multiple of 64 above 64)
   while activations are written with pitch cin: configs with such a channel count are refused at l2s_create, before
   any kernel could run, and the drop-in classes raise NotImplementedError.  No GPU is needed for any of this.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import vocoder_oracle as vo
import layer_reference as lr


def _chain(sd, h, cond):
    """Layer references chained on their own outputs, rounding off: the taps the oracle records."""
    w = lr.layer_weights(sd, None)
    out = {"conv_pre": lr.conv_pre(w, cond)}
    a = lr.activate(out["conv_pre"], None)
    x = None
    for i in range(len(h["upsample_rates"])):
        if i > 0:
            a = lr.activate(x, None)
        out[f"ups.{i}"] = lr.upsample(w, h, i, a)
        x = out[f"mrf.{i}"] = lr.mrf(w, h, i, out[f"ups.{i}"], None)
    out["wave"] = lr.head(w, x)
    return out


@pytest.mark.parametrize("variant", ["shipped", "unit_only"])
def test_layer_chain_reproduces_the_oracle(variant):
    if variant == "shipped":
        h = vo.shipped_config()
        sd = vo.init_state_dict(h, seed=1234, style="trained")
        code, mel, spkr = vo.synthetic_inputs(2, 16, seed=52)
        taps = {}
        wave = vo.mel_code_generator_forward(vo.fold_weight_norm(sd), h, code, mel, spkr, taps=taps)
        cond = lr.front_end(sd, h, code, mel, spkr)
    else:
        h = vo.unit_only_config()
        sd = vo.init_state_dict(h, seed=1234, style="trained", unit_only=True)
        g = torch.Generator().manual_seed(52)
        code = torch.randint(0, 200, (2, 12), generator=g)
        spkr = torch.randint(0, 200, (2, 1), generator=g)
        taps = {}
        wave = vo.code_generator_forward(vo.fold_weight_norm(sd), h, code, spkr, taps=taps)
        cond = lr.front_end(sd, h, code, spkr=spkr, unit_only=True)
    assert torch.equal(cond, taps["cond"].transpose(1, 2))
    got = _chain(sd, h, cond)
    names = ["conv_pre"] + [f"{kind}.{i}" for i in range(len(h["upsample_rates"])) for kind in ("ups", "mrf")]
    for name in names:
        ref = taps[name].transpose(1, 2)
        assert got[name].shape == ref.shape, name
        err = float((got[name] - ref).abs().max()) / max(1.0, float(ref.abs().max()))
        assert err <= 1e-12, (name, err)
    assert got["wave"].shape == wave[:, 0].shape
    assert float((got["wave"] - wave[:, 0]).abs().max()) <= 1e-12


def test_rounding_helpers_follow_the_device_conventions():
    one = 1.0
    tie = torch.tensor([one + 2.0 ** -11, -(one + 2.0 ** -11), one + 3 * 2.0 ** -12])
    # tf32 keeps 10 mantissa bits: 1 + 2^-11 is a tie (away from zero), 1 + 3 * 2^-12 rounds up
    assert lr.tf32_rna(tie).tolist() == [one + 2.0 ** -10, -(one + 2.0 ** -10), one + 2.0 ** -10]
    assert lr.tf32_trunc(tie).tolist() == [one, -one, one]
    # bf16: round to nearest even from the fp32 value
    assert lr.bf16(torch.tensor([one + 2.0 ** -8, one + 3 * 2.0 ** -8], dtype=torch.float64)).tolist() == [one, one + 2.0 ** -6]
    # the bf16 leaky-ReLU: slope bf16(0.1) = 0.10009765625 applied to the bf16 value, product rounded to bf16
    x = torch.randn(4096, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    a = lr.activate(x, "bf16")
    v = x.float().to(torch.bfloat16)
    assert torch.equal(a, torch.where(v > 0, v, v * torch.tensor(0.1).to(torch.bfloat16)).double())
    assert torch.equal(lr.bf16(a), a)
    assert float((a - F.leaky_relu(x, 0.1)).abs().max()) <= 2.0 ** -8 * float(x.abs().max())
    t = lr.activate(x, "tf32")
    assert torch.equal(lr.tf32_rna(t), t) and float((t - F.leaky_relu(x, 0.1)).abs().max()) <= 2.0 ** -11 * float(x.abs().max())
    assert torch.equal(lr.activate(x, None), F.leaky_relu(x, 0.1))


def _create(pkg, h, precision):
    lib = pkg._cabi.load()
    g = pkg.MelCodeGenerator(pkg.AttrDict(h))
    g.set_precision(precision)
    cfg = g._config()
    hnd = C.c_void_p()
    st = lib.l2s_create(C.byref(cfg), C.byref(hnd))
    msg = pkg._cabi.last_error(lib, hnd)
    lib.l2s_destroy(hnd)
    return st, msg


# stages 96 / 48 and 192 / 96 / 48: the 96-channel layers would read rows with pitch 128
PADDED = [(192, [5, 4], [11, 8], "resblocks.0.convs1.0"), (384, [5, 4, 4], [11, 8, 8], "resblocks.3.convs1.0")]
# stages 128 / 64 / 32 and 256 / 128 / 64 (the configs of the GPU layer-parity tests) and the shipped one
UNPADDED = [(256, [5, 4, 4], [11, 8, 8]), (512, [5, 4, 4], [11, 8, 8]), (512, [5, 4, 2, 2, 2], [11, 8, 4, 4, 4])]


@pytest.mark.parametrize("precision", ["bf16", "tf32", "fp32"])
def test_create_refuses_padded_channel_counts(pkg, precision):
    for c0, rates, ks, layer in PADDED:
        h = vo.shipped_config(upsample_initial_channel=c0, upsample_rates=rates, upsample_kernel_sizes=ks)
        st, msg = _create(pkg, h, precision)
        assert st == pkg._cabi.ERR_UNSUPPORTED, (c0, st, msg)
        assert layer in msg and "96 input channels" in msg and "multiples of 64" in msg, msg
        g = pkg.MelCodeGenerator(pkg.AttrDict(h))
        g.load_state_dict(vo.init_state_dict(h, seed=1, style="trained"), strict=True)
        g.eval()
        g.set_precision(precision)
        with pytest.raises(NotImplementedError, match=layer):
            g._engine(torch.device("cuda", 0))             # refused at l2s_create: no device is touched
    for c0, rates, ks in UNPADDED:
        h = vo.shipped_config(upsample_initial_channel=c0, upsample_rates=rates, upsample_kernel_sizes=ks)
        st, msg = _create(pkg, h, precision)
        assert st == pkg._cabi.OK, (c0, rates, msg)
