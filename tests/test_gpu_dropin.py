"""The drop-in boundary on the B200, exercised the way the reference's vocoder service uses it
(multi_input_vocoder/inference_server.py:85-146): a separate process runs `dropin.py <caller script>`, the caller does
`from models_multi_input import MelCodeGenerator` next to a sibling of that name, builds the generator from the JSON
config, loads a weight-normed checkpoint, vocodes the shipped lrs3 sample rows one at a time and writes int16 wav
files; they are compared with the oracle.  (The upstream repository is not part of this one, so the caller is the
restated tests/dropin_caller/inference_like.py; the unmodified reference script is run through the same launcher
by tests/test_dropin_cpu.py when L2S_REFERENCE_DIR names an upstream checkout.)"""
import os
import sys

import pytest

from test_dropin_cpu import CALLER, LAUNCHER, ROOT, _check_wavs, _run, make_job

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("precision,lsb", [("fp32", 1), ("bf16", 660)])
def test_service_call_sequence_through_the_launcher(pkg, tmp_path, precision, lsb):
    """fp32 mode: every sample within 1 int16 LSB of the fp64 oracle; bf16 mode: within the stated max-abs tolerance
    (2e-2 = 655 LSB; measured ~1e-2)."""
    tmp = str(tmp_path)
    fix = os.path.join(ROOT, "tests", "golden", "lrs3_handoff")
    cfg, ckpt, tsv, dct, sd, h = make_job(tmp, fix, precision=precision)
    out = os.path.join(tmp, "out")
    r = _run([sys.executable, LAUNCHER, CALLER, cfg, tsv, dct, "--checkpoint_file", ckpt, "--output_dir", out], cwd=tmp)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("wrote ") == 5
    _check_wavs(out, fix, sd, h, lsb=lsb)
