"""Layer-by-layer parity: every layer of the CUDA forward against an fp64 reference fed that layer's OWN device input.

The end-to-end tests compare waveforms with whole-tensor metrics, and the kernel-variant tests compare kernels with
each other; neither shows that one layer's arithmetic is right everywhere.  A single wrong row per utterance (a tile
tail, a halo row, a phase-major block with its bias added twice) keeps a tensor SNR near 49 dB.  Here each layer is
recomputed in fp64 (tests/layer_reference.py) from the debug tap of its input, so errors do not compound, and every
ELEMENT must sit within a tolerance far below the end-to-end noise.

Per case (config, precision, kernel knobs, batch, frames): forwards stopped after every MRF stage give the `ups` and
`mrf` taps of each stage (forwards are deterministic, so the stopped forwards form one chain), a full forward gives the
waveform, and the first stopped forward the `cond` and `conv_pre_act` taps.  Compared:
  cond          vs the oracle's cond (fp64, from the test inputs); the pad lanes (cin .. cin_pad) must be exactly 0
  conv_pre_act  vs act(conv_pre(device cond)), act = leaky_relu(0.1) as the epilogue stores it
  ups.i         vs ConvTranspose1d on the device conv_pre_act (i = 0) or act(device mrf.{i-1}) (the kernels write the
                activated copy from the same fp32 value as the raw one)
  mrf.i         vs the stage's ResBlocks + branch mean on the device ups.i
  wave          vs leaky_relu(0.01) -> conv_post -> tanh on the device mrf of the last stage
Operands are rounded where the kernels store them (bf16 / tf32 weights and conv input activations; see
tests/layer_reference.py), so what remains is fp32 summation order and one-ulp flips of re-rounded intermediates.

Metrics.  Activations stored in bf16 (`cond`, `conv_pre_act` in bf16 mode) or tf32 (`conv_pre_act` in tf32 mode): the
device value must be ref rounded to that format or a neighbouring value (see _neighbour), at most NEIGHBOUR_FRAC of
the elements may differ from the rounded reference, and elements beyond one step (fp32 cancellation on tiny values)
must stay within `*_far` x rms(ref).  Everything else: max over elements of |dev - ref| / rms(ref).

Tolerances (TOL) against the maxima measured over all 146 cases on a B200 (1000 W power limit); every tolerance is at
most 4x its measured maximum (profiles/r03_layer_parity.txt):
  mode  layer              tolerance   measured
  bf16  cond / conv_pre    off the rounded ref <= 0.4 % of elements (measured 0.009 % / 0.11 %)
        cond_far           2e-7        5.05e-8
        conv_pre_far       1.4e-5      3.64e-6
        ups                4e-5        1.12e-5
        mrf                8e-3        2.67e-3
        wave               1e-5        2.91e-6
  tf32  cond               1e-6        3.09e-7
        conv_pre           off the rounded ref <= 6.5 % of elements (measured 1.72 %)
        conv_pre_far       5e-5        1.46e-5
        ups                8e-5        2.14e-5
        mrf                1.6e-3      4.47e-4
        wave               1.2e-5      3.01e-6
  fp32  cond               1e-6        3.09e-7
        conv_pre           6e-5        1.62e-5
        ups                3e-5        8.24e-6
        mrf                1e-5        2.63e-6
        wave               8e-6        2.28e-6
The bf16 bounds sit far below what a localized defect produces: a row of one branch without its bias (|b| up to 0.05
in the "trained" init, activations of rms 0.5 - 1) moves the MRF output by ~1e-2 x rms, a missing tap by more.

tf32 mode: weights and every activated copy are rounded to nearest tf32 before the tensor core sees them, except the
conditioning tensor, which conv_pre reads as plain fp32.  Measured on conv_pre over every tf32 case: emulating
kind::tf32 by TRUNCATING those operands leaves at most 1.72 % of the tf32 outputs off the rounded reference (rms error
9.1e-5 of rms(ref)); rounding them to nearest leaves 67 % off (rms error 6.1e-4).  The tensor core truncates, and
the reference does the same (TF32_COND).

The fp64 references run on the GPU (torch conv1d / conv_transpose1d in float64).  Wall time of this file on a B200:
about 2 minutes (114 s for the 146 cases).
"""
import pytest
import torch

from oracle import vocoder_oracle as vo
import layer_reference as lr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# per (mode, layer): the largest value seen by the cases of this run, printed at the end of the module
MEASURED = {}
TOL = {
    "bf16": dict(cond_far=2e-7, conv_pre_far=1.4e-5, ups=4e-5, mrf=8e-3, wave=1e-5),
    "tf32": dict(cond=1e-6, conv_pre_far=5e-5, ups=8e-5, mrf=1.6e-3, wave=1.2e-5),
    "fp32": dict(cond=1e-6, conv_pre=6e-5, ups=3e-5, mrf=1e-5, wave=8e-6),
}
NEIGHBOUR_FRAC = {"bf16": 4e-3, "tf32": 6.5e-2}
TF32_COND = "trunc"     # how kind::tf32 treats fp32 operands with more than 10 mantissa bits (measured, see above)

CONFIGS = {
    "shipped": dict(h=vo.shipped_config(), seed=1234),
    "unit_only": dict(h=vo.unit_only_config(), seed=1234, unit_only=True),
    # ConvTranspose1d with k > 3u (padding larger than the stride)
    "k_gt_3u": dict(h=vo.shipped_config(upsample_rates=[2, 4, 2], upsample_kernel_sizes=[8, 16, 4], upsample_initial_channel=128,
                                        resblock_kernel_sizes=[3, 7], resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]]), seed=7),
    # ResBlock kernel sizes 5 / 9, two (even) dilations per branch
    "k5_9": dict(h=vo.shipped_config(upsample_rates=[4, 4, 2], upsample_kernel_sizes=[8, 8, 4], upsample_initial_channel=128,
                                     resblock_kernel_sizes=[5, 9], resblock_dilation_sizes=[[1, 2], [2, 4]]), seed=11),
    # last stage C = 32 (stages 128 / 64 / 32) and C = 64 (256 / 128 / 64): the other waveform heads
    "c32": dict(h=vo.shipped_config(upsample_initial_channel=256, upsample_rates=[5, 4, 4], upsample_kernel_sizes=[11, 8, 8]), seed=5),
    "c64": dict(h=vo.shipped_config(upsample_initial_channel=512, upsample_rates=[5, 4, 4], upsample_kernel_sizes=[11, 8, 8]), seed=6),
}

# bf16 kernel families (knob settings) of the shipped config
FAMILIES = {
    "default": {},
    "pack0": {"pack": 0},                                   # tap-by-tap whole-ResBlock kernels on C <= 64
    "pk_all": {"pk_chan": 16 | 32 | 64},                    # time-packed kernel on every narrow stage
    "pk_none": {"pk_chan": 0},
    "steps": {"fuse_branch": 0},                            # fused c1 -> c2 step kernels everywhere
    "unfused": {"fuse_branch": 0, "fuse_pairs": 0},         # one tcgen05 conv per launch
    "skew": {"res_skew": 1, "res_mode": 2, "pack": 0},      # skewed whole-ResBlock schedule
    "simt": {"force_simt": 1},                              # CUDA-core bf16 convs
    "post_tile": {"post_rows": 0},                          # staged-tile waveform head
    "front_split": {"front_fuse": 0},                       # separate speaker projection kernel
}
DEFAULT_KNOBS = {"stop_after_stage": -1, "pack": 1, "pk_chan": 32, "fuse_branch": 1, "fuse_pairs": 1, "res_skew": 0,
                 "res_mode": 0, "force_simt": 0, "post_rows": 1, "front_fuse": 1}

MATRIX = [(c, p, "default") for c in CONFIGS for p in ("bf16", "tf32", "fp32")]
MATRIX += [("shipped", "bf16", f) for f in FAMILIES if f != "default"]
MATRIX += [(c, "bf16", "post_tile") for c in ("c32", "c64")]
# tile tails, utterances shorter than a tile, several tiles per utterance, batches that do not divide the grid
SHAPES = [(1, 2), (1, 10), (3, 34), (5, 66), (2, 514)]
CASES = [(c, p, f, b, t) for c, p, f in MATRIX for b, t in SHAPES] + [("shipped", "bf16", "default", 1, 1300)]


@pytest.fixture(scope="module")
def gens(pkg):
    cache = {}

    def get(cfg, precision):
        if (cfg, precision) not in cache:
            spec = CONFIGS[cfg]
            uo = spec.get("unit_only", False)
            sd = vo.init_state_dict(spec["h"], seed=spec["seed"], style="trained", unit_only=uo)
            g = (pkg.CodeGenerator if uo else pkg.MelCodeGenerator)(pkg.AttrDict(spec["h"]))
            g.load_state_dict(sd, strict=True)
            g.eval()
            g.remove_weight_norm()
            g.set_precision(precision)
            cache[(cfg, precision)] = (g.to(DEV), sd)
        return cache[(cfg, precision)]

    yield get
    if MEASURED:
        print("\n[layer-parity] maxima over the cases run (mode, layer): value")
        for k in sorted(MEASURED):
            print(f"[layer-parity]   {k[0]:5s} {k[1]:10s} {MEASURED[k]:.3e}")


def _inputs(cfg, batch, frames):
    if CONFIGS[cfg].get("unit_only"):
        g = torch.Generator().manual_seed(71 + frames)
        return dict(code=torch.randint(0, 200, (batch, frames), generator=g), spkr=torch.randint(0, 200, (batch, 1), generator=g))
    code, mel, spkr = vo.synthetic_inputs(batch, frames, seed=71 + frames)
    return dict(code=code, mel=mel, spkr=spkr)


def _record(mode, layer, value):
    MEASURED[(mode, layer)] = max(MEASURED.get((mode, layer), 0.0), value)


def _where(err, frames_per_utt):
    """(b, t, c) of the largest element of a (B, L, C) error tensor, and a description of where that is."""
    idx = int(torch.argmax(err))
    b, rem = divmod(idx, err.shape[1] * err.shape[2])
    t, c = divmod(rem, err.shape[2])
    return (b, t, c), (f"(b={b}, t={t}, c={c}): {t} rows from the utterance start, {frames_per_utt - 1 - t} from its end, "
                       f"t mod 128 = {t % 128}")


def _normalized(dev, ref, what, tol, fails):
    """max |dev - ref| / rms(ref) over every element; appends a failure message naming the worst element."""
    dev = dev.to(ref.device, torch.float64)
    if dev.dim() == 2:
        dev, ref = dev.unsqueeze(-1), ref.unsqueeze(-1)
    assert dev.shape == ref.shape, what
    rms = float(ref.pow(2).mean().sqrt())
    err = (dev - ref).abs() / rms
    m = float(err.max()) if torch.isfinite(dev).all() else float("inf")
    if not m <= tol:
        (b, t, c), where = _where(torch.nan_to_num(err, nan=float("inf")), ref.shape[1])
        fails.append(f"{what}: max |dev - ref| / rms(ref) = {m:.3e} > {tol:.1e} at {where}; dev {float(dev[b, t, c]):.6e}, "
                     f"ref {float(ref[b, t, c]):.6e}, rms(ref) {rms:.3e}")
    return m


def _steps(dev, ref, fmt):
    """Distance in storage-format steps (bf16 or tf32) between the device value and ref rounded to that format
    (sign-magnitude bit patterns mapped onto ordered integers)."""
    def ordered(x):
        if fmt == "bf16":
            u = x.float().to(torch.bfloat16).view(torch.int16).long()
            mag = u & 0x7FFF
        else:
            u = lr.tf32_rna(x.float()).view(torch.int32).long()
            mag = (u & 0x7FFFFFFF) >> 13
        return torch.where(u < 0, -mag, mag)
    return (ordered(dev) - ordered(ref)).abs()


def _neighbour(dev, ref, what, fmt, far_tol, fails):
    """Low-precision storage (bf16 activations, tf32 activated copies): every device value is ref rounded to the storage
    format or a neighbouring value of it -- up to two steps for negative bf16 values, whose activation rounds twice
    (bf16(x), then bf16(x) * bf16(0.1)), so that one step of bf16(x) can become two steps of the output -- and at most
    NEIGHBOUR_FRAC of the elements differ from the rounded reference at all.  Exception: elements that fp32 accumulation
    puts further from a tiny reference value (cancellation), as long as |dev - ref| <= far_tol * rms(ref).
    Returns (fraction of elements not equal to the rounded reference, max |dev - ref| / rms(ref) beyond the allowance)."""
    dev = dev.to(ref.device)
    steps = _steps(dev, ref, fmt)
    rms = float(ref.pow(2).mean().sqrt())
    frac = float((steps > 0).double().mean())
    allowed = torch.where(ref < 0, 2 if fmt == "bf16" else 1, 1)
    far = steps > allowed
    far_err = float(((dev.double() - ref).abs() / rms)[far].max()) if bool(far.any()) else 0.0
    if far_err > far_tol or frac > NEIGHBOUR_FRAC[fmt]:
        (b, t, c), where = _where(torch.where(far, (dev.double() - ref).abs(), torch.zeros_like(ref)), ref.shape[1])
        fails.append(f"{what}: {int(far.sum())} elements beyond one {fmt} step of the reference, the worst "
                     f"|dev - ref| / rms(ref) = {far_err:.3e} (<= {far_tol:.1e}) at {where}; dev {float(dev[b, t, c]):.6e}, "
                     f"ref {float(ref[b, t, c]):.6e}; {100 * frac:.3f} % of the elements off the rounded reference "
                     f"(<= {100 * NEIGHBOUR_FRAC[fmt]:.2f} %)")
    return frac, far_err


@pytest.mark.parametrize("cfg,precision,family,batch,frames", CASES, ids=[f"{c}-{p}-{f}-{b}x{t}" for c, p, f, b, t in CASES])
def test_layer_parity(pkg, gens, cfg, precision, family, batch, frames):
    spec = CONFIGS[cfg]
    h, uo = spec["h"], spec.get("unit_only", False)
    g, sd = gens(cfg, precision)
    lib = pkg._cabi.load()
    inp = _inputs(cfg, batch, frames)
    dinp = {k: v.to(DEV) for k, v in inp.items()}
    rates, n = h["upsample_rates"], len(h["upsample_rates"])
    chans = [h["upsample_initial_channel"] >> (i + 1) for i in range(n)]
    lens = [frames * int(torch.tensor(rates[:i + 1]).prod()) for i in range(n)]
    in_dim = h["model_in_dim"]
    cin_pad = (in_dim + 63) // 64 * 64                      # make_conv: cin > 64 is padded to a multiple of 64
    taps = {}
    try:
        for k, v in FAMILIES[family].items():
            assert lib.l2s_debug_set(k.encode(), v) == 0, k
        for i in range(n):
            lib.l2s_debug_set(b"stop_after_stage", i)
            g(**dinp)
            if i == 0:
                taps["cond"] = g.debug_tap("cond", (batch, frames, cin_pad), DEV)
                taps["conv_pre_act"] = g.debug_tap("conv_pre_act", (batch, frames, h["upsample_initial_channel"]), DEV)
            taps[f"ups.{i}"] = g.debug_tap("ups", (batch, lens[i], chans[i]), DEV)
            taps[f"mrf.{i}"] = g.debug_tap("mrf", (batch, lens[i], chans[i]), DEV)
        lib.l2s_debug_set(b"stop_after_stage", -1)
        wave = g(**dinp)[:, 0].cpu()
    finally:
        for k, v in DEFAULT_KNOBS.items():
            lib.l2s_debug_set(k.encode(), v)

    mode = precision
    rmode = {"fp32": None, "tf32": "tf32", "bf16": "bf16_simt" if family == "simt" else "bf16"}[mode]
    w = lr.to_device(lr.layer_weights(sd, rmode), DEV)
    tol, fails, line = TOL[mode], [], []
    # ---- conditioning front end: the oracle's cond from the test's own inputs; pad lanes exactly zero
    ref_cond = lr.front_end(sd, h, **inp, unit_only=uo).to(DEV)
    cond = taps["cond"].to(DEV)
    if cin_pad > in_dim and not bool((cond[..., in_dim:] == 0).all()):
        fails.append(f"cond: pad lanes {in_dim}..{cin_pad - 1} are not all zero")
    cond = cond[..., :in_dim]
    if mode == "bf16":
        frac, far = _neighbour(cond, ref_cond, "cond", "bf16", tol["cond_far"], fails)
        _record(mode, "cond_nb", frac)
        _record(mode, "cond_far", far)
        line.append(f"cond nb {frac:.2e} far {far:.2e}")
    else:
        e = _normalized(cond, ref_cond, "cond", tol["cond"], fails)
        _record(mode, "cond", e)
        line.append(f"cond {e:.2e}")
    # ---- conv_pre on the device cond operand
    operand = cond.double()
    if mode == "tf32":
        # conv_pre reads the fp32 cond values: both emulations of the tensor core's tf32 conversion are measured and
        # printed (the evidence for TF32_COND), the one in TF32_COND is the reference
        for name, fn in (("trunc", lr.tf32_trunc), ("rna", lr.tf32_rna)):
            ref = lr.activate(lr.conv_pre(w, fn(cond).double()), mode)
            steps = _steps(taps["conv_pre_act"].to(DEV), ref, "tf32")
            off = float((steps > 0).double().mean())
            rel = float((taps["conv_pre_act"].to(DEV).double() - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt())
            _record(mode, f"pre_{name}_off", off)
            _record(mode, f"pre_{name}_rms", rel)
            line.append(f"conv_pre[{name}] off {off:.2e} rms {rel:.2e} max steps {int(steps.max())}")
        operand = (lr.tf32_trunc if TF32_COND == "trunc" else lr.tf32_rna)(cond).double()
    ref_pre = lr.activate(lr.conv_pre(w, operand), rmode)
    if mode in ("bf16", "tf32"):
        frac, far = _neighbour(taps["conv_pre_act"], ref_pre, "conv_pre_act", mode, tol["conv_pre_far"], fails)
        _record(mode, "conv_pre_nb", frac)
        _record(mode, "conv_pre_far", far)
        line.append(f"conv_pre nb {frac:.2e} far {far:.2e}")
    else:
        e = _normalized(taps["conv_pre_act"], ref_pre, "conv_pre_act", tol["conv_pre"], fails)
        _record(mode, "conv_pre", e)
        line.append(f"conv_pre {e:.2e}")
    # ---- upsamplers and MRF stages, each on its own device input
    for i in range(n):
        a = taps["conv_pre_act"].to(DEV).double() if i == 0 else lr.activate(taps[f"mrf.{i - 1}"].to(DEV), rmode)
        e_u = _normalized(taps[f"ups.{i}"], lr.upsample(w, h, i, a), f"ups.{i}", tol["ups"], fails)
        e_m = _normalized(taps[f"mrf.{i}"], lr.mrf(w, h, i, taps[f"ups.{i}"].to(DEV), rmode), f"mrf.{i} (C = {chans[i]})",
                          tol["mrf"], fails)
        _record(mode, "ups", e_u)
        _record(mode, "mrf", e_m)
        line.append(f"ups.{i} {e_u:.2e} mrf.{i} {e_m:.2e}")
    # ---- waveform head on the device output of the last stage
    e = _normalized(wave, lr.head(w, taps[f"mrf.{n - 1}"].to(DEV)), "wave", tol["wave"], fails)
    _record(mode, "wave", e)
    line.append(f"wave {e:.2e}")
    print(f"[layer-parity] {cfg} {precision} {family} {batch}x{frames}: " + ", ".join(line))
    assert not fails, "\n".join(fails)
