"""Shared helpers for the parity tests (tests may import oracle/)."""
import json
import os
import re

import numpy as np
import torch

from oracle import spexplus as ospex
from wesep_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# SI-SDR is invariant to a DC shift of the estimate, so d(loss)/d(decoder bias) is exactly 0 in exact arithmetic:
# both sides only hold fp32 round-off there (|g| ~ 1e-5..1e-4, different with every reduction order, i.e. with the
# CPU's thread count and vector width) and a relative comparison is meaningless.
ZERO_GRAD = re.compile(r"decoder\.decoder_1d_\d\.bias$")


def load_fixture(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    return z, meta


def load_layouts():
    """{"spex/<fuse type>" | "bsrnn/<fuse type>/multi_fuse=<bool>": [[key, shape], ...]}: the reference state_dict layouts
    (tests/golden/make_golden_layouts.py)."""
    return json.loads(str(np.load(os.path.join(GOLDEN, "state_dict_layouts.npz"))["layouts"]))


def cfg_from_args(args):
    cfg = dict(ospex.DEFAULT_CFG)
    for k in ("N", "L", "B", "H", "P", "X", "R", "spk_emb_dim", "spk_fuse_type", "multi_task", "spksInTrain"):
        if k in args:
            cfg[k] = args[k]
    return cfg


def fixture_inputs(meta, dtype=torch.float32, device="cpu"):
    cfg = cfg_from_args(meta["args"])
    sd = ospex.make_state_dict(cfg, dtype=dtype, device="cpu")
    synth.fill_state_dict_(sd, seed=meta["wseed"])
    sd = {k: v.to(device) for k, v in sd.items()}
    batch = synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=meta["dseed"], dtype=dtype)
    batch = {k: v.to(device) for k, v in batch.items()}
    return cfg, sd, batch


def rel_l2(a, b):
    a = a.double().flatten()
    b = b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def score_case(seed, snr_db, T):
    """Seeded (est, ref, mix) fp32 triple for the scoring fixtures: ref = speech-like coloured noise with a DC
    offset, mix = ref + interferer, est = 0.7 * ref + residual at `snr_db`."""
    rng = np.random.default_rng(seed)
    ref = rng.standard_normal(T).astype(np.float32) * 0.1 + 0.01
    itf = rng.standard_normal(T).astype(np.float32) * 0.12
    err = rng.standard_normal(T).astype(np.float32)
    scale = np.linalg.norm(ref) / max(np.linalg.norm(err), 1e-12) * 10 ** (-snr_db / 20)
    est = (0.7 * ref + err * scale).astype(np.float32)
    mix = (ref + itf).astype(np.float32)
    return est, ref, mix


def frontend_waves(seed, lengths):
    """Seeded fp32 utterances for the data front end fixtures: AR(1)-coloured noise at speech-like level, distinct
    gain and DC offset per utterance."""
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(lengths):
        e = rng.standard_normal(n)
        x = np.empty(n)
        acc = 0.0
        for j in range(n):
            acc = 0.9 * acc + e[j]
            x[j] = acc
        out.append((x * (0.02 + 0.01 * i) + 0.003 * (i - 1)).astype(np.float32))
    return out


# name, seed, utterance lengths (speaker 0 first), chunk length, use_random_snr
MIX_CASES = [("two_0db", 3, [20000, 17003], 8000, False),
             ("two_snr", 4, [9000, 30011], 8000, True),
             ("short_tiled", 5, [3000, 8000], 8000, True),          # utterance shorter than the chunk: tiled
             ("three_snr", 6, [12000, 8001, 15000], 6001, True)]
# name, seed, samples, dtype of the wave handed to compute_fbank (soundfile gives float64, torchaudio.load float32)
FBANK_CASES = [("f64_4s", 8, 64000, np.float64), ("f32_1s", 9, 16400, np.float32), ("one_frame", 10, 400, np.float64),
               ("odd", 11, 12345, np.float64)]


class SqTiny(torch.nn.Module):
    """Stand-in speaker encoder for the BSRNN_Multi fixtures (the real one, wespeaker's, is an external package): energy per
    mel bin averaged over frames, then Linear.  Returns wespeaker's (dummy, embedding) tuple.  Plain torch: test scaffolding on
    both sides, not part of the path under test."""

    def __init__(self, feat_dim=80, embed_dim=256, **kw):
        super().__init__()
        self.fc = torch.nn.Linear(feat_dim, embed_dim)

    def forward(self, x):  # x [n, frames, feat_dim]
        return torch.zeros((), device=x.device), self.fc((x ** 2).mean(1))
