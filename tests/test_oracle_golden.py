"""CPU: the oracle restatement (oracle/*.py) vs golden outputs of the REAL reference
(tests/golden/*.npz, produced by tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import losses as olosses
from oracle import optim as ooptim
from oracle import spexplus as ospex
from tests.util import ZERO_GRAD, fixture_inputs, load_fixture

SMALL_CASES = ["spex_small_train", "spex_small_eval", "spex_small_n1", "spex_small_FiLM", "spex_small_multiply",
               "spex_small_additive", "spex_small_concat"]


def _run(name, backward):
    z, meta = load_fixture(name)
    cfg, sd, b = fixture_inputs(meta)
    params = {}
    if backward:
        for k, v in sd.items():
            if v.is_floating_point() and "running_" not in k:
                v.requires_grad_(True)
                params[k] = v
    bufs = {}
    out = ospex.convtasnet_forward(sd, cfg, b["wav_mix"], b["spk_embeds"], training=meta["train"], buffers_out=bufs)
    tgt = b["wav_targets"][:, :out[0].shape[-1]]
    loss, parts = olosses.train_loss(out, tgt, b["spk_label"], multi_task=cfg["multi_task"])
    sub = meta["subsample"]
    for i in range(3):
        ref = torch.from_numpy(z[f"out{i}"])
        got = out[i].detach()[..., ::sub]
        assert got.shape == ref.shape
        assert torch.allclose(got, ref, rtol=1e-3, atol=2e-5), (name, i, float((got - ref).abs().max()))
        s = olosses.sisdr_per_row(out[i].detach().double(), tgt.double()).numpy()
        assert np.max(np.abs(s - z[f"sisdr_rows{i}"])) <= 0.01, (name, i)   # dB, north-star tolerance
    if len(out) > 3:
        assert torch.allclose(out[3].detach(), torch.from_numpy(z["out3"]), rtol=1e-3, atol=1e-4)
    assert abs(float(loss) - float(z["loss"])) <= 1e-3 * abs(float(z["loss"])) + 1e-3
    if backward and meta["backward"]:
        loss.backward()
        for k, p in params.items():
            gn = float(p.grad.double().norm())
            ref = float(z["gnorm/" + k])
            if ZERO_GRAD.search(k):
                assert gn <= 1e-3 and ref <= 1e-3, (name, k, gn, ref)
                continue
            assert abs(gn - ref) <= 2e-3 * ref + 1e-6, (name, k, gn, ref)
            if ("g/" + k) in z:
                g = torch.from_numpy(z["g/" + k])
                assert (p.grad - g).norm() <= 2e-3 * g.norm() + 1e-6, (name, k)
    if meta["train"]:
        for k, v in bufs.items():
            assert torch.allclose(v, torch.from_numpy(z["buf/" + k]), rtol=1e-3, atol=1e-5), (name, k)


@pytest.mark.parametrize("name", SMALL_CASES)
def test_oracle_small(name):
    _run(name, backward=True)


def test_oracle_full_cfg1_eval():
    """BASELINE config 1: Spex+ forward + SI-SNR on one 2-speaker 4 s mixture (n=2)."""
    _run("spex_full_cfg1_eval", backward=False)


@pytest.mark.slow
def test_oracle_full_cfg1_train():
    _run("spex_full_cfg1_train", backward=True)


def test_optim_golden():
    z = np.load("tests/golden/optim.npz")
    n = 5
    params = [torch.from_numpy(z[f"p0_{i}"].copy()) for i in range(n)]
    m = [torch.zeros_like(p) for p in params]
    v = [torch.zeros_like(p) for p in params]
    for step in range(3):
        grads = [torch.from_numpy(z[f"g{step}_{i}"].copy()) for i in range(n)]
        norms = ooptim.clip_gradients(grads, 5.0)
        assert np.allclose(norms, z[f"norms{step}"], rtol=1e-5)
        ooptim.adam_step(params, grads, m, v, step + 1, float(z["lrs"][step]))
        for i in range(n):
            assert torch.allclose(params[i], torch.from_numpy(z[f"p{step + 1}_{i}"]), rtol=2e-5, atol=1e-7)


def test_sched_golden():
    z = np.load("tests/golden/sched.npz")
    for it, lr in zip(z["its"], z["lrs"]):
        mine = ooptim.exponential_decrease_lr(int(it), 150 * 1000)
        assert abs(mine - lr) <= 1e-12 + 1e-9 * lr


def test_sisnr_cross_check():
    """restated auraloss SISDRLoss vs in-tree cal_SISNR formula: <= 2e-6 dB (SURVEY App. B)."""
    z = np.load("tests/golden/sisnr.npz")
    for snr, a, c in z["rows"]:
        assert abs(a - c) < 1e-4
    rng = np.random.default_rng(3)
    t = rng.standard_normal(4000)
    x = 0.3 * t + 0.1 * rng.standard_normal(4000)
    a = float(olosses.sisdr_per_row(torch.from_numpy(x)[None], torch.from_numpy(t)[None])[0])
    c = float(olosses.cal_sisnr_numpy(t, x))
    assert abs(a - c) < 1e-6


def test_score_golden():
    """oracle/score.py (cal_SISNR / cal_SISNRi restated) vs the REAL reference functions' outputs
    (tests/golden/score.npz, make_golden_score.py): same fp32 numpy arithmetic -> <= 2e-5 dB; the fp64 evaluation
    is the value the CUDA kernel (fp64 moments) is held to."""
    from oracle import score as oscore
    from tests.util import score_case
    z = np.load("tests/golden/score.npz")
    for seed, snr, T, s, d, s64 in z["rows"]:
        est, ref, mix = score_case(int(seed), float(snr), int(T))
        a, b = oscore.cal_sisnri(est, ref, mix)
        assert abs(a - s) <= 2e-5 and abs(b - d) <= 2e-5
        a64 = oscore.cal_sisnr(est.astype(np.float64), ref.astype(np.float64))
        assert abs(a64 - s64) <= 1e-9
        assert abs(a64 - s) <= 5e-5          # fp32 numpy vs fp64: the reference's own rounding noise


def test_score_peak_rule():
    """infer.py:124-129: scale every row to 0.9 peak only if every row has a positive sample."""
    from oracle import score as oscore
    x = torch.tensor([[0.5, -2.0, 1.0], [-0.25, 0.1, -0.05]])
    y = oscore.peak_rule(x)
    assert np.allclose(np.abs(y).max(axis=1), 0.9)
    x2 = x.clone()
    x2[1] = -x2[1].abs()
    assert np.array_equal(oscore.peak_rule(x2), x2.numpy())


def test_frontend_mix_golden():
    """oracle/frontend.py random_chunk + snr_mixer vs the REAL reference processors (frontend_mix.npz): same torch CPU
    ops in the same order -> bit-exact."""
    from oracle import frontend as ofe
    from tests.util import MIX_CASES, frontend_waves
    z = np.load("tests/golden/frontend_mix.npz")
    for name, seed, lens, T, _ in MIX_CASES:
        waves = frontend_waves(seed, lens)
        chunks = [torch.from_numpy(ofe.random_chunk(w, T, int(c)))[None] for w, c in zip(waves, z[name + "/c0"])]
        mix, spk = ofe.snr_mixer(chunks, list(z[name + "/snr"]))
        assert np.array_equal(mix.numpy()[0], z[name + "/mix"]), name
        for i, s in enumerate(spk):
            assert np.array_equal(s.numpy()[0], z[name + f"/spk{i}"]), (name, i)


def test_frontend_fbank_golden():
    """oracle/frontend.py fbank (restated torchaudio.compliance.kaldi.fbank + CMN, fp64) vs the REAL reference
    compute_fbank + apply_cmvn outputs."""
    from oracle import frontend as ofe
    from tests.util import FBANK_CASES, frontend_waves
    z = np.load("tests/golden/frontend_fbank.npz")
    for name, seed, n_samp, dtype in FBANK_CASES:
        w = frontend_waves(seed, [n_samp])[0]
        got = ofe.fbank(w)
        ref = z[name]
        assert got.shape == ref.shape, name
        tol = 1e-9 if dtype == np.float64 else 2e-4        # the fp32 reference run carries its own rounding
        assert np.abs(got - ref).max() <= tol, (name, np.abs(got - ref).max())
