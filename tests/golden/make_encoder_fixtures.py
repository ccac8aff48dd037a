"""Generates the perception-encoder fixtures (run in the BUILD container, where /root/reference exists):

  encoder_weights.npz   every Keras array of /root/reference/encoder_files/new_gripper_encoder/model.h5 (read by h5min)
  encoder_config.json   its config.yaml (network / encoding_dim) + the last row of history.csv
  golden_encoder.npz    encodings of 8 seeded synthetic depth scenes by the float64 oracle (oracle/encoder_ref.py) and
                        the restated auto-encoder's reconstruction MSE on 64 scenes (the sanity anchor)
  encoder_model_h5_skeleton.npz
                        model.h5 with every weight payload cut out (24 KB of HDF5 structure), the offsets the payloads were
                        cut from and the SHA-256 of the whole file: with encoder_weights.npz it rebuilds model.h5 byte for byte

    python tests/golden/make_encoder_fixtures.py
"""
import csv
import hashlib
import json
import os
import struct
import sys

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import b200grasp  # noqa: E402,F401
from b200grasp import h5min, synth  # noqa: E402
from b200grasp.encoders import keras_encoder_arrays  # noqa: E402
from oracle import encoder_ref as E  # noqa: E402

SRC = "/root/reference/encoder_files/new_gripper_encoder"
OUT = os.path.dirname(os.path.abspath(__file__))

w = h5min.load_keras_weights(os.path.join(SRC, "model.h5"))
np.savez_compressed(os.path.join(OUT, "encoder_weights.npz"), **{k.replace("/", "__"): v for k, v in w.items()})

raw = open(os.path.join(SRC, "model.h5"), "rb").read()
cuts = []
for k, v in w.items():
    b = np.ascontiguousarray(v, "<f4").tobytes()
    o = raw.find(b)
    # the payload occurs once in the file, at an address a layout message names
    assert o >= 0 and raw.find(b, o + 1) < 0 and struct.pack("<Q", o) in raw, k
    cuts.append((o, k))
cuts.sort()
for (o, k), (nxt, _) in zip(cuts, cuts[1:]):
    assert o + w[k].nbytes <= nxt, k            # no two payloads overlap
keep, pos = [], 0
for o, k in cuts:
    keep.append(raw[pos:o])
    pos = o + w[k].nbytes
keep.append(raw[pos:])
np.savez_compressed(os.path.join(OUT, "encoder_model_h5_skeleton.npz"), skeleton=np.frombuffer(b"".join(keep), np.uint8),
                    offsets=np.array([o for o, _ in cuts], np.int64), names=np.array([k for _, k in cuts]),
                    sha256=hashlib.sha256(raw).hexdigest())
cfg = yaml.safe_load(open(os.path.join(SRC, "config.yaml")))
hist = list(csv.DictReader(open(os.path.join(SRC, "history.csv"))))
json.dump({"network": cfg["network"], "encoding_dim": cfg["encoding_dim"], "alpha": cfg.get("alpha", 0.1),
           "history_last": {k: float(v) for k, v in hist[-1].items()},
           "shapes": {k: list(v.shape) for k, v in sorted(w.items())}},
          open(os.path.join(OUT, "encoder_config.json"), "w"), indent=1)

strides = [l["strides"] for l in cfg["network"]]
arr = keras_encoder_arrays(w, len(strides))
dec = [(w["dense_2/kernel"], w["dense_2/bias"])] + [(w[f"conv2d_{i}/kernel"], w[f"conv2d_{i}/bias"]) for i in (4, 5, 6)]
imgs = synth.make_depth_scenes(8, seed=11)
z64 = E.encode(imgs, arr, strides, cfg.get("alpha", 0.1), torch.float64)
big = synth.make_depth_scenes(64, seed=12)
rec = E.decode(E.encode(big, arr, strides), dec, strides, (8, 8, 32))
mse = float(((rec - big) ** 2).mean())
np.savez_compressed(os.path.join(OUT, "golden_encoder.npz"), z=z64, recon_mse=mse, img_energy=float((big ** 2).mean()))
print("encodings", z64.shape, "recon mse", mse, "image energy", float((big ** 2).mean()), "history", hist[-1])
