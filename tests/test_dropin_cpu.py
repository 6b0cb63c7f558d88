"""The drop-in boundary as the reference's own scripts reach it: `from models_multi_input import MelCodeGenerator`
(multi_input_vocoder/inference.py:28, inference_server.py:28).  CPU side: import resolution, the launcher's
precedence over the script-directory sibling, and -- when L2S_REFERENCE_DIR names a checkout of the upstream
lip2speech-unit repository -- the UNMODIFIED reference inference.py executed through the launcher up to the generator
call, which on a machine without a B200 must fail loudly (there is no CPU fallback)."""
import json
import os
import shutil
import subprocess
import sys

import pytest
import torch

from oracle import vocoder_oracle as vo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "lip2speech-unit_b200")
LAUNCHER = os.path.join(PKG_DIR, "dropin.py")
CALLER = os.path.join(ROOT, "tests", "dropin_caller", "inference_like.py")
STUBS = os.path.join(ROOT, "tests", "stubs")
REF = os.path.abspath(os.environ["L2S_REFERENCE_DIR"]) if os.environ.get("L2S_REFERENCE_DIR") else None   # upstream checkout
REF_SCRIPT = os.path.join(REF, "multi_input_vocoder", "inference.py") if REF else None


def _run(cmd, env_extra=None, cwd=None):
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    env.update(env_extra or {})
    return subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=cwd, timeout=600)


def test_top_level_import_like_the_reference_scripts(pkg):
    """PYTHONPATH shadowing (a script that has no sibling of that name): the module must import as a top-level
    module, without a parent package (ADVICE r1: `from . import _cabi` used to raise here)."""
    r = _run([sys.executable, "-c",
              "from models_multi_input import MelCodeGenerator, CodeGenerator, AttrDict; import models_multi_input as m; print(m.__file__)"],
             env_extra={"PYTHONPATH": PKG_DIR}, cwd="/")
    assert r.returncode == 0, r.stderr
    assert os.path.samefile(r.stdout.strip().splitlines()[-1], os.path.join(PKG_DIR, "models_multi_input.py"))


def test_launcher_beats_the_script_directory_sibling(pkg):
    """A script's own directory is sys.path[0], ahead of PYTHONPATH, so the reference's sibling models_multi_input.py
    would always win; the launcher registers the B200 module in sys.modules first.  The caller sits next to a decoy
    sibling that raises when imported."""
    r = _run([sys.executable, CALLER, "cfg", "tsv", "dict", "--checkpoint_file", "x", "--probe"], env_extra={"PYTHONPATH": PKG_DIR})
    assert r.returncode != 0 and "decoy" in r.stderr                      # without the launcher the sibling wins
    r = _run([sys.executable, LAUNCHER, CALLER, "cfg", "tsv", "dict", "--checkpoint_file", "x", "--probe"])
    assert r.returncode == 0, r.stderr
    assert os.path.samefile(r.stdout.strip().splitlines()[-1], os.path.join(PKG_DIR, "models_multi_input.py"))


def make_job(tmp, root, precision=None):
    """config JSON + random-init checkpoint in the reference's format ({'generator': weight-normed state dict},
    train.py:198-207) + a manifest whose first line points at `root`."""
    h = vo.shipped_config()
    cfg = dict(h)
    cfg.update(code_hop_size=320, mel_hop_size=160, n_fft=1024, hop_size=256, win_size=1024, sampling_rate=16000, fmin=0,
               fmax=8000, fmax_for_loss=None, segment_size=8960, num_mels=80)
    cfg.pop("text_supervision", None)              # the scripts set it from the environment (inference_server.py:110)
    if precision:
        cfg["precision"] = precision
    cfg_path = os.path.join(tmp, "config.json")
    with open(cfg_path, "w") as f:
        json.dump(cfg, f)
    sd = vo.init_state_dict(h, seed=1234, style="trained")
    ckpt = os.path.join(tmp, "g_00000001")
    torch.save({"generator": sd}, ckpt)
    fix = os.path.join(ROOT, "tests", "golden", "lrs3_handoff", "label")
    os.makedirs(os.path.join(tmp, "label"), exist_ok=True)
    with open(os.path.join(fix, "test.tsv")) as f:
        rows = f.read().splitlines()
    with open(os.path.join(tmp, "label", "test.tsv"), "w") as f:
        f.write("\n".join([root] + rows[1:]) + "\n")
    shutil.copy(os.path.join(fix, "test.unt"), os.path.join(tmp, "label", "test.unt"))
    shutil.copy(os.path.join(fix, "dict.unt.txt"), os.path.join(tmp, "label", "dict.unt.txt"))
    return cfg_path, ckpt, os.path.join(tmp, "label", "test.tsv"), os.path.join(tmp, "label", "dict.unt.txt"), sd, h


@pytest.mark.skipif(not (REF_SCRIPT and os.path.isfile(REF_SCRIPT)), reason="set L2S_REFERENCE_DIR to an upstream lip2speech-unit checkout")
def test_unmodified_reference_inference_py_through_the_launcher(pkg, tmp_path):
    """`python dropin.py <reference>/multi_input_vocoder/inference.py cfg manifest dict --checkpoint_file ... --debug`:
    the reference's argument parsing, parse_manifest, MelCodeDataset, init_worker (MelCodeGenerator(h).to(device),
    load_state_dict of the weight-normed checkpoint, eval, remove_weight_norm) and the first dataset item all run
    unmodified; the class they got is the B200 one.  Without a GPU the generator call must raise (no CPU fallback);
    with one, the written wav files must match the oracle."""
    tmp = str(tmp_path)
    cfg, ckpt, tsv, dct, sd, h = make_job(tmp, os.path.join(REF, "datasets", "lrs3"), precision="fp32")
    out = os.path.join(tmp, "out")
    r = _run([sys.executable, LAUNCHER, REF_SCRIPT, cfg, tsv, dct, "--checkpoint_file", ckpt, "--output_dir", out, "--debug", "-n", "-1"],
             env_extra={"PYTHONPATH": STUBS}, cwd=tmp)
    log = r.stdout + r.stderr
    assert "Initializing Inference Process" in log and "Complete." in log, log      # main() and load_checkpoint() ran
    assert "decoy" not in log
    if not torch.cuda.is_available():
        assert r.returncode != 0
        assert os.path.join("lip2speech-unit_b200", "models_multi_input.py") in log, log   # the traceback passes through OUR forward
        assert "no CPU fallback" in log, log
        return
    assert r.returncode == 0, log
    _check_wavs(out, os.path.join(REF, "datasets", "lrs3"), sd, h, lsb=1)


def _check_wavs(out_dir, root, sd, h, lsb):
    import numpy as np
    from scipy.io import wavfile
    import __graft_entry__ as ge
    ho = ge.load_package().hand_off
    fix = os.path.join(ROOT, "tests", "golden", "lrs3_handoff")
    _, rows = ho.parse_manifest(os.path.join(fix, "label", "test.tsv"))
    code_dict = ho.load_code_dict(os.path.join(fix, "label", "dict.unt.txt"))
    w = vo.fold_weight_norm(sd)
    n_checked = 0
    for r in rows:
        feats, n = ho.load_item(fix, r, code_dict)
        ref = vo.mel_code_generator_forward(w, h, torch.from_numpy(feats["code"]).unsqueeze(0), torch.from_numpy(feats["mel"]).unsqueeze(0),
                                            torch.from_numpy(feats["spkr"]).unsqueeze(0), dtype=torch.float64)
        want = (ref.squeeze() * 32768.0).numpy().astype("int16")
        path = os.path.join(out_dir, ho.output_name(r) + ".wav")
        assert os.path.isfile(path), path
        rate, got = wavfile.read(path)
        assert rate == 16000 and got.shape == want.shape
        diff = int(np.abs(got.astype(np.int32) - want.astype(np.int32)).max())
        print(f"[dropin] {ho.output_name(r)}: {n} samples, max |int16 diff| vs oracle {diff} LSB")
        assert diff <= lsb, (path, diff)
        n_checked += 1
    assert n_checked == 5
