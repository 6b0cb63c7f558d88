"""Benchmark of the multi_input_vocoder generator forward on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step is one forward of the hot path over one batch of synthetic utterances
(BASELINE.md section 4 distribution, seed 52) with random-init weights of the shipped
vocoder config (seed 1234).  Per-GPU workload = BASELINE.json configs[1]:
16 utterances x 4 s (T = 400 mel frames, U = 200 units), bf16 tensor-core mode.
Utterances are independent, so N GPUs run N such batches with no collective on
the data path (weak scaling).  torch.distributed is used for the start barrier and
the max-over-ranks of the device time only, over the gloo (CPU) backend: NCCL is
never initialised.

Prints ONE JSON line (rank 0).  `value` = audio-seconds generated per second with
inputs resident in HBM; `e2e` = the same through the public class with pinned host
inputs copied in and the waveform copied out every step.  `sustained` = the same
device-resident loop run back to back for >= 3 s (clocks and power sampled), the only
figure compared with the sustained tensor peak.  `extra` = the other BASELINE
configs through the public API: cfg3 (256 x 8 s split over the N ranks, strong
scaling) and cfg5 (64 x 6 s split over the ranks, multi-input vs unit-only).

--dump-outputs DIR writes the waveform the last timed step returned on rank 0, (16, 1, 64000) float32, as
DIR/waveform.npy.  Inputs and weights are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH, FRAMES = 16, 400          # configs[1]: 16 x 4 s
SR, HOP = 16000, 160
L2_MB = 126
REF_TREE = "/root/reference"     # only exists in the build container; optional everywhere


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(burst=float(d["bf16_tflops"]), sustained=float(d.get("bf16_tflops_sustained") or d["bf16_tflops"]),
                    hbm=float(d["hbm_gbs"]), src="MEASURED_PEAKS.json")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons sampled DURING the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def summary(self, t0=None, t1=None):
        sm, mx, pw, reasons = [], [], [], set()
        for ts, r in list(self.rows):
            if (t0 is not None and ts < t0) or (t1 is not None and ts > t1):
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(self.NAMES, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
            try:
                pw.append(float(r[6]))
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_median": statistics.median(pw) if pw else None}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        return self.summary()


def ncu_traffic():
    """dram read+write bytes per launch of the dominant kernels, from the committed ncu metrics pass (or None)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            return float(d["traffic_bytes_per_launch_avg"]), d["source"]
        except Exception:
            continue
    return None, None


# ----------------------------------------------------------------------------- CPU reference leg
def import_reference_classes():
    """The reference's own classes, when its tree is present (the build container): imported unmodified, with the
    absent matplotlib stubbed exactly as tests/golden/make_golden.py does.  None on the GPU box (no /root/reference)."""
    if not os.path.isdir(os.path.join(REF_TREE, "multi_input_vocoder")):
        return None
    try:
        m = types.ModuleType("matplotlib")
        m.use = lambda *a, **k: None
        sys.modules.setdefault("matplotlib", m)
        sys.modules.setdefault("matplotlib.pylab", types.ModuleType("matplotlib.pylab"))
        for sub in ("multi_input_vocoder", "speech-resynthesis"):
            pth = os.path.join(REF_TREE, sub)
            if pth not in sys.path:
                sys.path.insert(0, pth)
        saved = sys.modules.pop("models_multi_input", None)     # never the drop-in: this leg times the REFERENCE
        try:
            import importlib
            mod = importlib.import_module("models_multi_input")
            from utils import AttrDict
        finally:
            ref_mod = sys.modules.pop("models_multi_input", None)
            if saved is not None:
                sys.modules["models_multi_input"] = saved
        if os.path.commonpath([os.path.abspath(ref_mod.__file__), REF_TREE]) != REF_TREE:
            return None
        return mod.MelCodeGenerator, AttrDict
    except Exception:
        return None


def cpu_reference(seconds_budget=12.0):
    """The reference's CPU path on a bounded sample of the workload: 4 s utterances one at a time (the reference's own
    inference loop is batch 1, which is also its fastest CPU shape), fp32, all host threads, until ~seconds_budget.
    kind "reference": the reference's own MelCodeGenerator (only where /root/reference exists); kind "port": the
    oracle restatement (the same ATen operators, bit-comparable results; the reference tree cannot travel to the GPU box)."""
    from oracle import vocoder_oracle as vo
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    h = vo.shipped_config()
    sd = vo.init_state_dict(h, seed=1234, style="ref")
    code, mel, spkr = vo.synthetic_inputs(BATCH, FRAMES, seed=52)
    ref = import_reference_classes()
    if ref is not None:
        cls, attr = ref
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            g = cls(attr(dict(h)))
            g.load_state_dict(sd, strict=True)
            g.eval()
            g.remove_weight_norm()

        def run(i):
            return g(code=code[i:i + 1], mel=mel[i:i + 1], spkr=spkr[i:i + 1])
        kind = "reference"
    else:
        w = vo.fold_weight_norm(sd)

        def run(i):
            return vo.mel_code_generator_forward(w, h, code[i:i + 1], mel[i:i + 1], spkr[i:i + 1], dtype=torch.float32)
        kind = "port"
    with torch.no_grad():
        run(0)                                       # warm-up
        n, t0 = 0, time.perf_counter()
        while True:
            run(n % BATCH)
            n += 1
            el = time.perf_counter() - t0
            if el >= seconds_budget or n >= 4 * BATCH:
                break
    audio = n * FRAMES * HOP / SR
    return {"value": audio / el, "unit": "audio-s/s", "cores": threads, "kind": kind,
            "sample": f"{n} utterances x 4 s (T=400), batch 1, fp32, torch {torch.__version__} CPU, {el:.1f} s"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    res, total_audio, total_t = None, 0.0, 0.0
    per_step_budget = max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    for i in range(args.warmup + args.steps):
        res = cpu_reference(per_step_budget)
        if i >= args.warmup:
            n = int(res["sample"].split()[0])
            a = n * FRAMES * HOP / SR
            total_audio += a
            total_t += a / res["value"]
    value = total_audio / total_t
    res["value"] = value
    line = {"impl": "reference", "metric": "audio-sec generated/sec (16 kHz)", "value": value, "unit": "audio-s/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg2: 16 x 4 s utterances (T=400,U=200), multi_input_aug.json generator, "
                                   "random-init seed 1234; each step a bounded batch-1 sample of it on the host cores"},
            "cpu_baseline": res,
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------- helpers of our arm
def make_generator(pkg, vo, dev, precision, unit_only=False):
    h = vo.unit_only_config() if unit_only else vo.shipped_config()
    sd = vo.init_state_dict(h, seed=1234, style="ref", unit_only=unit_only)
    gen = (pkg.CodeGenerator if unit_only else pkg.MelCodeGenerator)(pkg.AttrDict(h))
    gen.load_state_dict(sd, strict=True)
    gen.eval()
    gen.remove_weight_norm()
    gen.set_precision(precision)
    return gen.to(dev), h


def pipeline_pass(pkg, gen, dev, batches, outs, passes, sync_all):
    """`passes` timed passes over `batches` (pinned host tensors) through HostPipeline with int16 waveforms back; one
    untimed pass first.  Returns device ms per pass."""
    pipe = pkg.HostPipeline(gen, dev)
    for b, o in zip(batches, outs):
        pipe.submit(*b, o)
    pipe.finish()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(passes):
        for b, o in zip(batches, outs):
            pipe.submit(*b, o)
    pipe.s_out.synchronize()
    e1.record()
    sync_all()
    pipe.finish()
    return e0.elapsed_time(e1) / passes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sustained loop and the cfg3 / cfg5 extras")
    ap.add_argument("--knob", action="append", default=[], help="debug knob k=v passed to l2s_debug_set")
    ap.add_argument("--layers", action="store_true", help="also print a per-launch time table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the waveform of the last timed step to DIR/waveform.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch.distributed as dist
    from oracle import vocoder_oracle as vo      # weights / synthetic inputs / cpu_baseline leg only
    import __graft_entry__ as ge

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # The CPU baseline is a rank-0, N = 1 figure: under torchrun the other ranks would spin in a barrier on the same
    # host cores while it runs, so it is skipped there (the N = 1 line carries it).
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference(12.0)
    if world > 1:
        dist.init_process_group("gloo")          # barrier + max-over-ranks only; the data path has no collective (no NCCL)
    ge.build()
    pkg = ge.load_package()
    lib = pkg._cabi.load()
    for kv in args.knob:
        k, v = kv.split("=")
        assert lib.l2s_debug_set(k.encode(), int(v)) == 0, kv

    gen, h = make_generator(pkg, vo, dev, args.precision)

    # every rank vocodes its own 16 x 4 s shard (seed differs per rank)
    code_h, mel_h, spk_h = vo.synthetic_inputs(BATCH, FRAMES, seed=52 + rank)
    code_h, mel_h, spk_h = code_h.pin_memory(), mel_h.pin_memory(), spk_h.pin_memory()
    code, mel, spk = code_h.to(dev), mel_h.to(dev), spk_h.to(dev)
    audio_per_step = BATCH * FRAMES * HOP / SR
    flops_per_step = vo.algorithmic_flops_per_frame(h) * BATCH * FRAMES

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    sampler = ClockSampler(local_rank)
    sampler.start()                     # keeps sampling through warm-up, the timed regions and the extras
    for _ in range(args.warmup):
        y = gen(code=code, mel=mel, spkr=spk)
    launches_per_step = gen.launch_count(BATCH, FRAMES, dev)
    ws_bytes = lib.l2s_workspace_bytes(gen._engine(dev).handle, BATCH, FRAMES)

    # ---- device-resident timed region
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_region0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        y = gen(code=code, mel=mel, spkr=spk)
    ev1.record()
    sync_all()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "waveform.npy"), y.cpu().numpy())
    # host time to ISSUE one step (no synchronisation): if it approaches ms_per_step the path is launch bound
    t_h0 = time.perf_counter()
    for _ in range(args.steps):
        y = gen(code=code, mel=mel, spkr=spk)
    host_ms = (time.perf_counter() - t_h0) * 1e3 / args.steps
    torch.cuda.synchronize()

    # ---- end to end through the public API: every step copies its inputs from pinned host memory to the device and
    # its waveform back to pinned host memory.  HostPipeline (dispatch.py) is the call a user with many batches makes:
    # the copies of neighbouring steps overlap the forward (two copy streams, double-buffered device inputs).
    out_h = [torch.empty((BATCH, 1, FRAMES * HOP), dtype=torch.float32).pin_memory() for _ in range(2)]
    pipe = pkg.HostPipeline(gen, dev)
    for i in range(4):
        pipe.submit(code_h, mel_h, spk_h, out_h[i & 1])
    pipe.finish()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        pipe.submit(code_h, mel_h, spk_h, out_h[i & 1])
    pipe.s_out.synchronize()
    e1.record()
    sync_all()
    ms_e2e = e0.elapsed_time(e1)
    pipe.finish()
    if not torch.equal(out_h[(args.steps - 1) & 1], y.cpu()):
        raise RuntimeError("end-to-end pipeline output differs from the device-resident forward")
    # short steps: keep the GPU under the same load until nvidia-smi has delivered a few samples
    t_end = time.time() + 4.0
    while len(sampler.rows) < 8 and time.time() < t_end:
        for _ in range(10):
            gen(code=code, mel=mel, spkr=spk)
        torch.cuda.synchronize()
    t_region1 = time.time()
    clocks = sampler.summary(t_region0, t_region1)
    if not clocks["samples"]:
        clocks = sampler.summary()
    h2d = code_h.numel() * 8 + mel_h.numel() * 4 + spk_h.numel() * 4
    d2h = out_h[0].numel() * 4

    # ---- sustained: the same device-resident loop back to back for >= 3 s (what the sustained tensor peak is measured like)
    sustained = None
    if not args.no_extra:
        n_sus = max(args.steps, int(3200.0 / (ms / args.steps)) + 1)
        sync_all()
        t_s0 = time.time()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(n_sus):
            gen(code=code, mel=mel, spkr=spk)
        s1.record()
        sync_all()
        t_s1 = time.time()
        ms_sus = max_over_ranks([s0.elapsed_time(s1)])[0]
        sustained = {"steps": n_sus, "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus,
                     "value": world * audio_per_step / (ms_sus / 1e3 / n_sus), "clocks": sampler.summary(t_s0 + 0.3, t_s1)}

    # ---- the other BASELINE configs through the public API (pinned host in, int16 waveform back), split over the ranks
    extra = None
    if not args.no_extra:
        extra = {}
        # cfg3: 256 x 8 s (T = 800) in total, strong scaling: rank r vocodes utterances r, r + N, ... in batches of <= 32
        mine = list(range(rank, 256, world))
        batches, outs = [], []
        for k in range(0, len(mine), 32):
            n_b = len(mine[k:k + 32])
            c3, m3, s3 = vo.synthetic_inputs(n_b, 800, seed=300 + rank * 16 + k // 32)
            batches.append((c3.pin_memory(), m3.pin_memory(), s3.pin_memory()))
            outs.append(torch.empty((n_b, 800 * HOP), dtype=torch.int16).pin_memory())
        ms3 = max_over_ranks([pipeline_pass(pkg, gen, dev, batches, outs, 3, sync_all)])[0]
        extra["cfg3"] = {"workload": f"256 x 8 s utterances (T=800) split over {world} rank(s), batches of <= 32, HostPipeline, int16 back",
                         "scaling": "strong", "ms": ms3, "value": 256 * 8.0 / (ms3 / 1e3), "unit": "audio-s/s",
                         "utterances_per_rank": len(mine)}
        # cfg5: 64 x 6 s in total, multi-input (T = 600) vs unit-only (U = 300, rates [5,4,4,2,2], speaker-id table)
        n5 = len(range(rank, 64, world))
        c5, m5, s5 = vo.synthetic_inputs(n5, 600, seed=500 + rank)
        b5 = [(c5.pin_memory(), m5.pin_memory(), s5.pin_memory())]
        o5 = [torch.empty((n5, 600 * HOP), dtype=torch.int16).pin_memory()]
        ms5 = max_over_ranks([pipeline_pass(pkg, gen, dev, b5, o5, 5, sync_all)])[0]
        gen_u, h_u = make_generator(pkg, vo, dev, args.precision, unit_only=True)
        gu = torch.Generator().manual_seed(600 + rank)
        cu = torch.randint(0, 200, (n5, 300), generator=gu, dtype=torch.int64).to(dev)
        su = torch.randint(0, 200, (n5, 1), generator=gu, dtype=torch.int64).to(dev)
        yu_h = torch.empty((n5, 300 * 320), dtype=torch.int16).pin_memory()

        def unit_step():
            yu = gen_u(code=cu, spkr=su)
            yu_h.copy_((yu.view(n5, -1) * 32768.0).clamp_(-32768, 32767).to(torch.int16), non_blocking=True)   # inference.py:79-81

        # warm up with the SAME loop body: torch loads the kernels of the int16 conversion lazily on their first use, and with
        # three bare forwards as warm-up those loads (12 ms of host time per step) landed in the timed region: 11.7 ms per step
        # at 8 utterances per rank where the forward takes 1.5 ms
        for _ in range(10):
            unit_step()
        sync_all()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        for _ in range(5):
            unit_step()
        u1.record()
        sync_all()
        msu = max_over_ranks([u0.elapsed_time(u1) / 5])[0]
        extra["cfg5"] = {"workload": f"64 x 6 s utterances split over {world} rank(s): multi-input (T=600, HostPipeline, int16 back) vs "
                                     "unit-only CodeGenerator (U=300, rates [5,4,4,2,2], device-resident ids, int16 back)",
                         "scaling": "strong", "utterances_per_rank": n5,
                         "multi_input": {"ms": ms5, "value": 64 * 6.0 / (ms5 / 1e3), "unit": "audio-s/s"},
                         "unit_only": {"ms": msu, "value": 64 * 6.0 / (msu / 1e3), "unit": "audio-s/s"}}
        del gen_u
        if world == 1:
            # cfg4: one 120 s stream (T = 12000) through vocode_long: chunks of 1000 frames + 24-frame halo per side, batched
            c4, m4, s4 = vo.synthetic_inputs(1, 12000, seed=400)
            c4, m4, s4 = c4.to(dev), m4.to(dev), s4.to(dev)
            for _ in range(2):
                y4 = pkg.vocode_long(gen, c4, m4, s4, core=1000)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(5):
                y4 = pkg.vocode_long(gen, c4, m4, s4, core=1000)
            f1.record()
            torch.cuda.synchronize()
            ms4 = f0.elapsed_time(f1) / 5
            extra["cfg4"] = {"workload": "one 120 s stream (T=12000) through dispatch.vocode_long: 12 chunks of 1000 frames + 24-frame halo per side in one "
                                         "batched forward, device-resident inputs, halo recompute not credited",
                             "ms": ms4, "value": 120.0 / (ms4 / 1e3), "unit": "audio-s/s"}

    # ---- per-launch times of one more forward (event pair per launch), for the roofline object
    lib.l2s_debug_set(b"layer_events", 1)
    gen(code=code, mel=mel, spkr=spk)
    torch.cuda.synchronize()
    import ctypes as C
    eng = gen._engine(dev)
    rows, i = [], 0
    while True:
        t, fl, nm = C.c_float(), C.c_double(), C.create_string_buffer(64)
        if lib.l2s_debug_layer_time(eng.handle, i, C.byref(t), C.byref(fl), nm, 64) != 0:
            break
        rows.append((nm.value.decode(), t.value, fl.value))
        i += 1
    lib.l2s_debug_set(b"layer_events", 0)
    final_clocks = sampler.stop()

    ms, ms_e2e = max_over_ranks([ms, ms_e2e])

    if rank == 0:
        pk = peaks()
        step_s = ms / 1e3 / args.steps
        conv_rows = [r for r in rows if r[2] > 0 and r[0] != "conv_post"]
        conv_ms = sum(r[1] for r in conv_rows)
        conv_flops = sum(r[2] for r in conv_rows)
        all_ms = sum(r[1] for r in rows)
        achieved = conv_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        stages = {}
        for name, t, fl in rows:
            if name.startswith("resblocks."):
                key = "mrf%d" % (int(name.split(".")[1].split()[0]) // len(h["resblock_kernel_sizes"]))
            elif name.startswith("ups."):
                key = "ups"
            else:
                key = name
            a = stages.setdefault(key, [0.0, 0.0])
            a[0] += t
            a[1] += fl
        stage_tbl = {k: {"ms": round(v[0], 4), "tflops": round(v[1] / (v[0] / 1e3) / 1e12, 1) if v[0] > 0 else 0.0}
                     for k, v in stages.items()}
        if args.layers:
            for name, t, fl in rows:
                sys.stderr.write(f"{name:28s} {t * 1e3:9.1f} us  {fl / max(t, 1e-9) / 1e9:8.1f} TFLOP/s\n")
        kernel = {"bf16": "pair_tc_kernel (fused ResBlock step, C >= 128) + respk_tc_kernel / res_tc_kernel (whole MRF stage / ResBlock, C <= 64) "
                          "+ conv_tc_kernel (conv_pre, ups): tcgen05 convolutions",
                  "tf32": "conv_tc_kernel (tcgen05 kind::tf32 tap-offset conv)", "fp32": "conv_simt_kernel"}[args.precision]
        traffic, traffic_src = ncu_traffic() if args.precision == "bf16" else (None, None)
        whole_tflops = flops_per_step / step_s / 1e12
        line = {
            "metric": "audio-sec generated/sec (16 kHz)",
            "value": world * audio_per_step / step_s,
            "unit": "audio-s/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms / args.steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": args.precision,
            "data": "synthetic",
            "config": {"workload": "cfg2 per GPU: 16 x 4 s utterances (T=400 mel frames, U=200 KM200 units, 256-d spk emb), "
                                   "multi_input_aug.json generator, random-init seed 1234",
                       "global_batch": world * BATCH, "audio_s_per_step": world * audio_per_step,
                       "parallelism": f"utterance-sharded x{world}, no collective (gloo barrier only, NCCL never initialised)",
                       "l2": f"no flush: per-step activation working set {ws_bytes / 2**20:.0f} MiB > {L2_MB} MB L2"},
            "tensor_tflops_whole_step": whole_tflops,
            "tensor_frac_whole_step_burst": whole_tflops / pk["burst"],
            "roofline": {"bound": "tensor", "kernel": kernel, "achieved": achieved, "peak": pk["burst"], "unit": "TFLOP/s",
                         "frac": achieved / pk["burst"], "frac_burst": achieved / pk["burst"],
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": pk["src"] + " bf16_tflops (burst): every launch is timed alone with its own CUDA event pair, in a "
                                                    f"{ms:.0f} ms region at {clocks.get('sm_mhz')} MHz; the sustained peak is only used for the >= 3 s loop (sustained.frac_sustained)",
                         "launches": len(conv_rows), "sum_launch_ms": round(conv_ms, 4), "all_launch_ms": round(all_ms, 4),
                         "algorithmic_gflop_per_step": conv_flops / 1e9, "per_stage": stage_tbl},
            "e2e": {"value": world * audio_per_step / (ms_e2e / 1e3 / args.steps), "unit": "audio-s/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps,
                    "api": "HostPipeline.submit(code, mel, spkr, out) per step: pinned host inputs -> device, MelCodeGenerator forward, fp32 waveform -> pinned host; copies of neighbouring steps overlap the forward"},
            "gpu_launches": launches_per_step * args.steps,
            "host_issue_ms_per_step": host_ms,
            "clocks": clocks,
        }
        if sustained is not None:
            sus_tflops = flops_per_step / (sustained["ms_per_step"] / 1e3) / 1e12
            sustained["tensor_tflops_whole_step"] = sus_tflops
            sustained["frac_sustained"] = sus_tflops / pk["sustained"]
            sustained["frac_burst"] = sus_tflops / pk["burst"]
            sustained["peaks"] = {"sustained": pk["sustained"], "burst": pk["burst"]}
            line["sustained"] = sustained
            line["roofline"]["frac_sustained"] = sustained["frac_sustained"]   # whole step, >= 3 s loop, vs the sustained peak
        if extra is not None:
            line["extra"] = extra
        line["clocks_whole_run"] = final_clocks
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        elif world > 1:
            line["cpu_baseline"] = {"skipped": "N > 1: the CPU baseline is a rank-0 figure of the N = 1 run (other ranks would share the host cores)"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
