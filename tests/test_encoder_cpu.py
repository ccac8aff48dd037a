"""Perception encoder (SURVEY section 8 row a12), CPU side: the model.h5 reader, the oracle against its committed golden
encodings, and the reconstruction anchor that ties the restated auto-encoder to the reference's training history."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import b200grasp  # noqa: F401
from b200grasp import h5min, synth
from b200grasp.encoders import keras_encoder_arrays
from oracle import encoder_ref as E
from tests.util import GOLD


def load_fixture():
    w = {k.replace("__", "/"): v for k, v in np.load(os.path.join(GOLD, "encoder_weights.npz")).items()}
    cfg = json.load(open(os.path.join(GOLD, "encoder_config.json")))
    return w, cfg


def test_fixture_inventory_matches_the_reference_graph():
    w, cfg = load_fixture()
    # encoders.py:87-128 with config.yaml's network: 3 encoder convs, Dense(100), Dense(2048), 2 decoder convs + output conv
    assert [tuple(w[f"conv2d_{i}/kernel"].shape) for i in range(1, 7)] == [
        (7, 7, 1, 32), (5, 5, 32, 32), (3, 3, 32, 32), (3, 3, 32, 32), (5, 5, 32, 32), (7, 7, 32, 1)]
    assert w["dense_1/kernel"].shape == (2048, 100) and w["dense_2/kernel"].shape == (100, 2048)
    assert sum(v.size for v in w.values()) == 484677
    assert cfg["encoding_dim"] == 100 and [l["strides"] for l in cfg["network"]] == [2, 2, 2]


def rebuild_model_h5(w):
    """The reference's model.h5, byte for byte: its stored HDF5 structure with the committed weights put back where they
    were cut out (tests/golden/make_encoder_fixtures.py), checked against the SHA-256 of the original file."""
    sk = np.load(os.path.join(GOLD, "encoder_model_h5_skeleton.npz"))
    skeleton, raw, s = sk["skeleton"].tobytes(), b"", 0
    for o, k in zip(sk["offsets"].tolist(), sk["names"].tolist()):
        n = o - len(raw)                                  # structure bytes in front of this payload
        raw += skeleton[s:s + n] + np.ascontiguousarray(w[k], "<f4").tobytes()
        s += n
    raw += skeleton[s:]
    assert hashlib.sha256(raw).hexdigest() == str(sk["sha256"])
    return raw


def test_h5_reader_reproduces_the_committed_weights(tmp_path):
    w, _ = load_fixture()
    h5 = tmp_path / "model.h5"
    h5.write_bytes(rebuild_model_h5(w))
    got = h5min.load_keras_weights(str(h5))
    assert sorted(got) == sorted(w)
    for k in w:
        assert got[k].dtype == np.float32 and np.array_equal(got[k], w[k]), k


def test_h5_reader_rejects_non_hdf5(tmp_path):
    p = tmp_path / "x.h5"
    p.write_bytes(b"not an hdf5 file at all")
    with pytest.raises(ValueError):
        h5min.H5File(str(p))


def test_same_padding_rule():
    # TF 'same': front pad = floor(total / 2)
    assert E.same_pad(64, 7, 2) == (2, 3) and E.same_pad(32, 5, 2) == (1, 2) and E.same_pad(16, 3, 2) == (0, 1)
    assert E.same_pad(16, 3, 1) == (1, 1) and E.same_pad(7, 3, 2) == (1, 1)


def test_oracle_reproduces_golden_encodings():
    w, cfg = load_fixture()
    strides = [l["strides"] for l in cfg["network"]]
    arr = keras_encoder_arrays(w, len(strides))
    g = np.load(os.path.join(GOLD, "golden_encoder.npz"))
    imgs = synth.make_depth_scenes(8, seed=11)
    z64 = E.encode(imgs, arr, strides, cfg["alpha"], torch.float64)
    np.testing.assert_allclose(z64, g["z"], rtol=1e-12, atol=1e-14)
    z32 = E.encode(imgs, arr, strides, cfg["alpha"], torch.float32)
    assert np.abs(z32 - g["z"]).max() <= 1e-4 * np.abs(g["z"]).max()


def test_reconstruction_anchor_against_training_history():
    """The only output-level evidence the reference offers: history.csv ends at val_loss 1.17e-3.  The restated
    encoder->decoder must reconstruct depth-like scenes at that error scale; a wrong padding side or flatten order
    raises it roughly tenfold (above the energy of the images themselves)."""
    w, cfg = load_fixture()
    strides = [l["strides"] for l in cfg["network"]]
    arr = keras_encoder_arrays(w, len(strides))
    dec = [(w["dense_2/kernel"], w["dense_2/bias"])] + [(w[f"conv2d_{i}/kernel"], w[f"conv2d_{i}/bias"]) for i in (4, 5, 6)]
    imgs = synth.make_depth_scenes(64, seed=12)
    rec = E.decode(E.encode(imgs, arr, strides), dec, strides, (8, 8, 32))
    mse = float(((rec - imgs) ** 2).mean())
    assert mse < 2.0 * cfg["history_last"]["val_loss"], mse
    swapped, orig = None, E.same_pad
    try:
        E.same_pad = lambda size, k, s: tuple(reversed(orig(size, k, s)))
        rec_bad = E.decode(E.encode(imgs, arr, strides), dec, strides, (8, 8, 32))
        swapped = float(((rec_bad - imgs) ** 2).mean())
    finally:
        E.same_pad = orig
    assert swapped > 5 * mse
