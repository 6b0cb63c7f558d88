"""The vocoder service's call sequence, restated so that it runs without the upstream repository.

Follows multi_input_vocoder/inference_server.py: module imports (:28), init() (:85-130: JSON -> AttrDict h,
h.code_dict_path, h.text_supervision from the environment, MelCodeGenerator(h).to(device),
torch.load(...)['generator'] -> load_state_dict, eval(), remove_weight_norm(), seeds) and inference() (:133-146:
one dataset item -> {k: torch.from_numpy(v).to(device).unsqueeze(0)} -> generator(**code) -> squeeze * 32768 ->
cpu int16 -> scipy wav under <output_dir>/pred_wav/<speaker>/<id>.wav), with the item built by the trimming rule of
dataset_multi_input.py:219-241.  It sits next to a decoy models_multi_input.py, the way the reference script sits
next to its own: only lip2speech-unit_b200/dropin.py makes the import below resolve to the B200 class.
"""
import argparse
import json
import os
import random
import sys

import numpy as np
import torch
from scipy.io.wavfile import write

from models_multi_input import MelCodeGenerator          # inference_server.py:28

MAX_WAV_VALUE = 32768.0                                   # speech-resynthesis/dataset.py:22


class AttrDict(dict):                                     # speech-resynthesis/utils.py:77-80
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.__dict__ = self


def read_rows(manifest, root_override):
    with open(manifest) as f:
        lines = [ln.rstrip("\n") for ln in f if ln.strip()]
    root = root_override or lines[0]
    with open(os.path.splitext(manifest)[0] + ".unt") as f:
        units = [ln.strip() for ln in f if ln.strip()]
    rows = []
    for ln, un in zip(lines[1:], units):
        cols = ln.split("\t")
        rows.append((os.path.join(root, cols[2]), int(cols[4]), un.split("|")[-1].split()))
    return rows


def load_item(row, code_dict, code_hop, mel_hop):
    wav_path, n_samples, toks = row
    code = np.array([code_dict[t] for t in toks if t in code_dict], dtype=np.int64)
    mel = np.load(wav_path.replace("/audio/", "/mel/")[:-4] + ".npy")
    n_code = min(n_samples // code_hop, code.shape[0])
    n_mel = min(n_samples // mel_hop, mel.shape[0])
    cut = min(n_mel * mel_hop, n_code * code_hop)
    feats = {"code": code[:cut // code_hop], "mel": np.ascontiguousarray(mel[:cut // mel_hop].T.astype(np.float32)),
             "spkr": np.load(wav_path.replace("/audio/", "/spk_emb/")[:-4] + ".npy")}
    return feats, wav_path


def main():
    p = argparse.ArgumentParser()
    p.add_argument("config_file")
    p.add_argument("input_code_file")
    p.add_argument("code_dict_path")
    p.add_argument("--output_dir", default="generated_files")
    p.add_argument("--checkpoint_file", required=True)
    p.add_argument("--root", default=None)
    p.add_argument("--probe", action="store_true", help="print where MelCodeGenerator came from and exit")
    a = p.parse_args()
    if a.probe:
        print(sys.modules[MelCodeGenerator.__module__].__file__)
        return
    device = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")
    with open(a.config_file) as f:
        h = AttrDict(json.loads(f.read()))
    h.code_dict_path = a.code_dict_path
    h.text_supervision = bool(int(os.environ.get("TEXT_SUPERVISION", 0)))
    generator = MelCodeGenerator(h).to(device)
    state_dict_g = torch.load(a.checkpoint_file, map_location="cpu")
    generator.load_state_dict(state_dict_g["generator"])
    os.makedirs(a.output_dir, exist_ok=True)
    generator.eval()
    generator.remove_weight_norm()
    random.seed(52); np.random.seed(52); torch.manual_seed(52)
    with open(a.code_dict_path) as f:
        code_dict = {ln.split()[0]: i for i, ln in enumerate(f) if ln.strip()}
    with torch.no_grad():
        for row in read_rows(a.input_code_file, a.root):
            feats, filename = load_item(row, code_dict, h.code_hop_size, h.mel_hop_size)
            code = {k: torch.from_numpy(v).to(device).unsqueeze(0) for k, v in feats.items()}
            y = generator(**code)
            if type(y) is tuple:
                y = y[0]
            audio = (y.squeeze() * MAX_WAV_VALUE).cpu().numpy().astype("int16")
            out = os.path.join(a.output_dir, os.path.join("pred_wav", *(filename.split("/")[-2:]))[:-4] + ".wav")
            os.makedirs(os.path.dirname(out), exist_ok=True)
            write(out, h.sampling_rate, audio)
            print("wrote", out)


if __name__ == "__main__":
    main()
