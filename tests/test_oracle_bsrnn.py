"""CPU: the pBSRNN oracle (oracle/bsrnn.py, SURVEY.md §8 rows a15-a21) vs golden outputs of the REAL reference
(tests/golden/bsrnn_*.npz from tests/golden/make_golden_bsrnn.py) and vs torch.stft / torch.istft."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import bsrnn as ob
from oracle import losses as olosses
from tests.util import load_layouts
from wesep_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SMALL = ["bsrnn_small_multiply", "bsrnn_small_additive_multi", "bsrnn_small_concat"]


def _state_dict_like(args):
    """Shapes of BSRNN(**args).state_dict() (joint_training False) without importing the reference: built from the
    constructor rules in wesep/models/bsrnn.py:16-36,55-69,244-282 and filled with the fixture's seed."""
    N = args["feature_dim"]
    E = args["spk_emb_dim"]
    R = args["num_repeat"]
    bands = ob.band_widths(args["sr"], args["win"])
    sd = {}
    for i, bw in enumerate(bands):
        sd[f"BN.{i}.0.weight"] = torch.empty(2 * bw)
        sd[f"BN.{i}.0.bias"] = torch.empty(2 * bw)
        sd[f"BN.{i}.1.weight"] = torch.empty(N, 2 * bw, 1)
        sd[f"BN.{i}.1.bias"] = torch.empty(N)

    def fuse(pre):
        in_f = E + N if args["spk_fuse_type"] == "concat" else E
        sd[pre + "fc.linear.weight"] = torch.empty(N, in_f)
        sd[pre + "fc.linear.bias"] = torch.empty(N)

    def resrnn(pre):
        sd[pre + "norm.weight"] = torch.empty(N)
        sd[pre + "norm.bias"] = torch.empty(N)
        for suf in ("", "_reverse"):
            sd[pre + "rnn.weight_ih_l0" + suf] = torch.empty(8 * N, N)
            sd[pre + "rnn.weight_hh_l0" + suf] = torch.empty(8 * N, 2 * N)
            sd[pre + "rnn.bias_ih_l0" + suf] = torch.empty(8 * N)
            sd[pre + "rnn.bias_hh_l0" + suf] = torch.empty(8 * N)
        sd[pre + "proj.weight"] = torch.empty(N, 4 * N)
        sd[pre + "proj.bias"] = torch.empty(N)

    def bsnet(pre):
        resrnn(pre + "band_rnn.")
        resrnn(pre + "band_comm.")

    sp = "separator.separation."
    if args["multi_fuse"]:
        for r in range(R):
            fuse(f"{sp}{2 * r}.")
            bsnet(f"{sp}{2 * r + 1}.")
    else:
        fuse(sp + "0.")
        for r in range(R):
            bsnet(f"{sp}{r + 1}.")
    for i, bw in enumerate(bands):
        sd[f"mask.{i}.0.weight"] = torch.empty(N)
        sd[f"mask.{i}.0.bias"] = torch.empty(N)
        sd[f"mask.{i}.1.weight"] = torch.empty(4 * N, N, 1)
        sd[f"mask.{i}.1.bias"] = torch.empty(4 * N)
        sd[f"mask.{i}.3.weight"] = torch.empty(4 * N, 4 * N, 1)
        sd[f"mask.{i}.3.bias"] = torch.empty(4 * N)
        sd[f"mask.{i}.5.weight"] = torch.empty(4 * bw, 4 * N, 1)
        sd[f"mask.{i}.5.bias"] = torch.empty(4 * bw)
    return sd


def _inputs(meta):
    b = synth.make_batch(meta["n"], T=meta["L"], Te=8, seed=meta["dseed"])
    rng = np.random.default_rng(meta["dseed"] + 77)
    emb = torch.from_numpy(rng.standard_normal((meta["n"], 256)).astype(np.float32))
    return b["wav_mix"], b["wav_targets"], emb


def _load(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    return z, json.loads(str(z["meta"]))


def test_state_dict_layout_matches_reference_order():
    """The key list (and order: optimizer state and checkpoints depend on it) equals the reference's, as stored from the
    reference BSRNN in tests/golden/state_dict_layouts.npz (tests/golden/make_golden_layouts.py)."""
    layouts = load_layouts()
    for fuse, mf in (("multiply", False), ("concat", True)):
        args = dict(spk_emb_dim=256, sr=16000, win=512, stride=128, feature_dim=16, num_repeat=2, use_spk_transform=False,
                    spk_fuse_type=fuse, multi_fuse=mf, joint_training=False)
        ref = [(k, tuple(s)) for k, s in layouts[f"bsrnn/{fuse}/multi_fuse={mf}"]]
        mine = _state_dict_like(args)
        assert [k for k, _ in ref] == list(mine.keys())
        assert all(s == tuple(mine[k].shape) for k, s in ref)


@pytest.mark.parametrize("L", [4000, 1023, 512])
def test_stft_istft_match_torch(L):
    g = torch.Generator().manual_seed(L)
    x = torch.randn(3, L, generator=g, dtype=torch.float64)
    w = torch.hann_window(512, dtype=torch.float32).double()
    re, im = ob.stft(x)
    S = torch.stft(x, n_fft=512, hop_length=128, window=w, return_complex=True)
    assert re.shape == S.real.shape
    assert float((re - S.real).abs().max()) < 1e-10 and float((im - S.imag).abs().max()) < 1e-10
    y = ob.istft(re, im, length=L)
    y2 = torch.istft(S, n_fft=512, hop_length=128, window=w, length=L)
    assert float((y - y2).abs().max()) < 1e-11
    assert float((y - x).abs().max()) < 1e-9          # perfect reconstruction (Hann, 75 % overlap)


def test_band_widths():
    b = ob.band_widths()
    assert b == [3] * 15 + [6] * 10 + [16] * 5 + [64] + [8] and sum(b) == 257 and len(b) == 32


def _run(name, backward):
    z, meta = _load(name)
    args = meta["args"]
    sd = synth.fill_state_dict_(_state_dict_like(args), seed=meta["wseed"])
    mix, tgt, emb = _inputs(meta)
    if backward:
        for v in sd.values():
            v.requires_grad_(True)
    est = ob.bsrnn_forward(sd, mix, emb, sr=args["sr"], win=args["win"], stride=args["stride"],
                           num_repeat=args["num_repeat"], spk_fuse_type=args["spk_fuse_type"], multi_fuse=args["multi_fuse"])
    ref = torch.from_numpy(z["out0"])
    got = est.detach()[..., ::meta["subsample"]]
    assert got.shape == ref.shape
    assert torch.allclose(got, ref, rtol=2e-3, atol=2e-6), (name, float((got - ref).abs().max()))
    s = olosses.sisdr_per_row(est.detach().double(), tgt.double()).numpy()
    assert np.max(np.abs(s - z["sisdr_rows0"])) <= 0.01, name             # dB, north-star tolerance
    loss = olosses.sisdr_loss(est, tgt)
    assert abs(float(loss) - float(z["loss"])) <= 1e-3
    if backward:
        loss.backward()
        for k, p in sd.items():
            ref_n = float(z["gnorm/" + k])
            gn = float(p.grad.double().norm())
            assert abs(gn - ref_n) <= 5e-3 * ref_n + 1e-7, (name, k, gn, ref_n)
            if ("g/" + k) in z:
                g = torch.from_numpy(z["g/" + k])
                assert (p.grad - g).norm() <= 5e-3 * g.norm() + 1e-7, (name, k)


@pytest.mark.parametrize("name", SMALL)
def test_oracle_bsrnn_small(name):
    _run(name, backward=True)


def test_oracle_bsrnn_recipe_size_forward():
    """bsrnn.yaml:48-55 network (feature 128, hidden 256, 6 repeats, 32 bands) on 1 s of audio, forward only."""
    _run("bsrnn_full_fwd_1s", backward=False)


@pytest.mark.parametrize("fuse,mf", [("multiply", False), ("concat", True), ("additive", False)])
def test_wesep_b200_bsrnn_state_dict_contract(fuse, mf):
    """wesep_b200.models.BSRNN registers its parameters under the reference's keys, shapes and ORDER (checkpoints,
    optimizer state); on CPU tensors its forward must refuse (there is no PyTorch fallback)."""
    from wesep_b200.models import get_model
    args = dict(spk_emb_dim=256, sr=16000, win=512, stride=128, feature_dim=16, num_repeat=2, use_spk_transform=False,
                spk_fuse_type=fuse, multi_fuse=mf, joint_training=False)
    m = get_model("BSRNN")(**args)
    want = _state_dict_like(args)
    got = m.state_dict()
    assert list(got.keys()) == list(want.keys())
    assert all(tuple(got[k].shape) == tuple(want[k].shape) for k in want)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 4000), torch.zeros(1, 256))


def test_wesep_b200_bsrnn_dft_bases_match_oracle_stft():
    """The constant analysis / synthesis matrices the CUDA path multiplies with (band-major spectrum rows, window folded
    in, models/bsrnn.py:_bases) reproduce the oracle's STFT / iSTFT when applied with plain matmuls on the CPU."""
    from wesep_b200.models import get_model
    m = get_model("BSRNN")(joint_training=False, use_spk_transform=False, feature_dim=16, num_repeat=1,
                           spk_fuse_type="multiply", multi_fuse=False)
    fwd_b, inv_b, offs, R, w2 = m._bases(torch.device("cpu"))
    assert R == 516 and fwd_b.shape == (516, 512) and inv_b.shape == (512, 516)
    L, win, hop = 3000, 512, 128
    x = torch.randn(2, L, generator=torch.Generator().manual_seed(3))
    re, im = ob.stft(x.double())
    T = re.shape[-1]
    xp = torch.cat([x[:, 1:257].flip(1), x, x[:, L - 257:L - 1].flip(1)], 1)
    idx = (torch.arange(T) * hop)[:, None] + torch.arange(win)[None, :]
    spec = torch.einsum("rk,btk->brt", fwd_b.double(), xp.double()[:, idx])         # [B, 516, T]
    lo = 0
    for o, bw in zip(offs, m.band_width):
        assert float((spec[:, o:o + bw] - re[:, lo:lo + bw]).abs().max()) < 1e-4
        assert float((spec[:, o + bw:o + 2 * bw] - im[:, lo:lo + bw]).abs().max()) < 1e-4
        lo += bw
    fr = torch.einsum("kr,brt->btk", inv_b.double(), spec)                          # windowed inverse-DFT frames
    n_out = win + hop * (T - 1)
    y = torch.zeros(2, n_out, dtype=torch.float64)
    env = torch.zeros(n_out, dtype=torch.float64)
    for t in range(T):
        y[:, t * hop:t * hop + win] += fr[:, t]
        env[t * hop:t * hop + win] += w2.double()
    rec = y[:, 256:256 + L] / env[256:256 + L]
    assert float((rec - x.double()).abs().max()) < 1e-4                             # analysis -> synthesis reconstructs
