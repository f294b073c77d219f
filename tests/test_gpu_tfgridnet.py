"""GPU: TF-GridNet (SURVEY.md §8 row a24) — the kernels of csrc/tfgridnet.cu, the attention on the pointwise GEMMs and the
LayerNorm + BLSTM + Linear paths vs fp64 restatements, and the whole model (forward, SISDR loss, every gradient) vs the golden
outputs of the REAL reference (tests/golden/tfgridnet_*.npz)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import losses as olosses
from oracle import tfgridnet as ot
from tests.test_gpu_dpccn import _act
from tests.test_gpu_kernels import check, rnd

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("H,E,T,Fq", [(4, 8, 37, 65), (2, 4, 9, 65), (1, 128, 21, 65), (1, 16, 5, 33)])
def test_head_ln(H, E, T, Fq):
    """PReLU + LayerNorm over (E, F) per (b, h, t): AllHeadPReLULayerNormalization4DCF (H > 1) and PReLU + LayerNormalization4DCF
    (H = 1, one slope); forward, gx and the three parameter gradients."""
    from wesep_b200 import ops
    B = 2
    x0 = rnd(B, H * E, T, Fq, seed=H + E, scale=1.3)
    al0 = (0.25 + 0.05 * rnd(H if H > 1 else 1, seed=1)).clone()
    ga0, be0 = 1 + 0.1 * rnd(1, H, E, 1, Fq, seed=2), 0.1 * rnd(1, H, E, 1, Fq, seed=3)
    g0 = rnd(B, H * E, T * Fq, seed=4)
    x = _act(x0)
    al, ga, be = (t.clone().requires_grad_(True) for t in (al0, ga0, be0))
    y = ops.HeadLnFn.apply(x, al, ga, be, H, T, Fq, 1e-5)
    y.backward(g0)
    x64 = x0.double().requires_grad_(True)
    a64, g64, b64 = (t.double().requires_grad_(True) for t in (al0, ga0, be0))
    sd = {"p.act.weight": a64.expand(H) if H > 1 else a64, "p.gamma": g64, "p.beta": b64}
    if H > 1:
        r = ot.all_head_prelu_ln(x64, sd, "p.", H, E, 1e-5).reshape(B, H * E, T, Fq)
    else:
        r = ot.ln_4dcf(ot.prelu(x64, a64, 1), {"p.gamma": g64.reshape(1, E, 1, Fq), "p.beta": b64.reshape(1, E, 1, Fq)}, "p.", 1e-5)
    r.backward(g0.double().reshape(B, H * E, T, Fq))
    check("y", y.detach(), r.detach().reshape(B, H * E, -1), 2e-5)
    check("gx", x.grad, x64.grad.reshape(B, H * E, -1), 5e-5)
    check("dgamma", ga.grad, g64.grad, 5e-5)
    check("dbeta", be.grad, b64.grad, 5e-5)
    check("dalpha", al.grad, a64.grad, 2e-4)


@pytest.mark.parametrize("R,C", [(40, 33), (1004, 1001)])
def test_softmax(R, C):
    from wesep_b200 import ops
    x0, g0 = rnd(1, R, C, seed=R, scale=3.0), rnd(1, R, C, seed=2)
    x = _act(x0)
    y = ops.SoftmaxFn.apply(x, 0.37)
    y.backward(g0)
    x64 = x0.double().requires_grad_(True)
    r = torch.softmax(0.37 * x64, -1)
    r.backward(g0.double())
    check("y", y.detach(), r.detach(), 1e-5)
    check("gx", x.grad, x64.grad, 2e-5)
    ld = y.stride(1)
    if ld > C:                                            # padding columns are zero (the matrix is a GEMM operand)
        assert not y.detach().as_strided((R, ld - C), (ld, 1), C).any()


def test_row_std():
    from wesep_b200 import ops
    x = rnd(5, 64000, seed=1, scale=0.1) + 0.02
    sd, inv = ops.row_std(x)
    ref = torch.std(x.double(), dim=1)
    check("std", sd, ref, 1e-6)
    check("inv", inv, 1 / ref, 1e-6)


@pytest.mark.parametrize("T,d,dv", [(33, 130, 520), (251, 520, 2080)])
def test_attention_rows(T, d, dv):
    """softmax(Q K / sqrt(d)) V for one (batch, head) on the pointwise GEMMs (T and d not multiples of 4 are padded)."""
    from wesep_b200 import ops
    Q0, K0, V0 = rnd(T, d, seed=1, scale=0.7), rnd(d, T, seed=2, scale=0.7), rnd(T, dv, seed=3)
    g0 = rnd(T, dv, seed=4)
    Qm, Kt, Vm = (t.clone().requires_grad_(True) for t in (Q0, K0, V0))
    o = ops.attention_rows(Qm, Kt, Vm)
    o.backward(g0)
    q64, k64, v64 = (t.double().requires_grad_(True) for t in (Q0, K0, V0))
    r = torch.softmax(q64 @ k64 / d ** 0.5, -1) @ v64
    r.backward(g0.double())
    check("out", o.detach(), r.detach(), 2e-5)
    check("dQ", Qm.grad, q64.grad, 5e-5)
    check("dK", Kt.grad, k64.grad, 5e-5)
    check("dV", Vm.grad, v64.grad, 5e-5)


@pytest.mark.parametrize("rows,C,S,Hd", [(70, 16, 65, 32), (130, 128, 21, 192)])
def test_layernorm_blstm_linear_path(rows, C, S, Hd):
    """intra / inter path of a GridNetBlock (gridnet_block.py:139-146): LayerNorm(C) -> BLSTM -> Linear + residual on
    [rows, C, S]; hidden 192 = the recipe's size on the cluster recurrence kernel."""
    from wesep_b200 import ops
    x0 = rnd(rows, C, S, seed=1)
    nw, nb = 1 + 0.1 * rnd(C, seed=2), 0.1 * rnd(C, seed=3)
    k = 1.0 / Hd ** 0.5
    names = ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]
    shapes = [(4 * Hd, C), (4 * Hd, Hd), (4 * Hd,), (4 * Hd,)]
    lstm0 = [k * rnd(*shp, seed=10 + i + 4 * j) for j in range(2) for i, shp in enumerate(shapes)]
    pw0, pb0 = rnd(C, 2 * Hd, seed=30, scale=0.1), 0.02 * rnd(C, seed=31)
    g0 = rnd(rows, C, S, seed=40)
    x = _act(x0)
    params = [t.clone().requires_grad_(True) for t in [nw, nb] + lstm0 + [pw0, pb0]]
    y = ops.res_rnn(x, params[0], params[1], params[2:10], params[10], params[11], layer_norm_eps=1e-5)
    y.backward(g0)
    p64 = [t.double().requires_grad_(True) for t in [nw, nb] + lstm0 + [pw0, pb0]]
    sd = {}
    for j, suf in enumerate(("", "_reverse")):
        for i, nme in enumerate(names):
            sd["r." + nme + suf] = p64[2 + 4 * j + i]
    x64 = x0.double().requires_grad_(True)
    xt = x64.transpose(1, 2)                                             # [rows, S, C]
    h = ot.blstm(ot.layer_norm_c(xt, p64[0], p64[1], 1e-5), sd, "r.")
    r = (h @ p64[10].t() + p64[11] + xt).transpose(1, 2)
    r.backward(g0.double())
    check("y", y.detach(), r.detach(), 2e-5)
    check("gx", x.grad, x64.grad, 1e-4)
    for i, (a, b) in enumerate(zip(params, p64)):
        check(f"param{i}", a.grad, b.grad, 3e-4)


def _golden_case(name, tol_g=3e-3):
    from wesep_b200 import ops, synth
    from wesep_b200.models import get_model
    z = np.load(os.path.join(GOLD, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    a = meta["args"]
    m = get_model("TFGridNet")(**a)
    ref_sd = ot.make_state_dict(n_layers=a["n_layers"], emb_dim=a["emb_dim"], hidden=a["lstm_hidden_units"], n_head=a["attn_n_head"],
                                approx_qk_dim=a["attn_approx_qk_dim"], n_fft=a["n_fft"], emb_ks=a["emb_ks"], emb_hs=a["emb_hs"])
    assert list(m.state_dict().keys()) == list(ref_sd.keys())
    assert all(m.state_dict()[k].shape == ref_sd[k].shape for k in ref_sd)
    synth.fill_state_dict_(m.state_dict(), seed=meta["wseed"])
    m = m.to(DEV).train()
    b = synth.make_batch(meta["n"], T=meta["L"], Te=8, seed=meta["dseed"], device=DEV)
    rng = np.random.default_rng(meta["dseed"] + 77)
    emb = torch.from_numpy(rng.standard_normal((meta["n"], 256)).astype(np.float32)).to(DEV)
    est, _ = m(b["wav_mix"], emb)
    ref = torch.from_numpy(z["out0"]).to(DEV)
    got = est.detach()[..., ::meta["subsample"]]
    assert got.shape == ref.shape
    check("est", got, ref, 1e-3)
    rows = olosses.sisdr_per_row(est.detach().double(), b["wav_targets"].double()).cpu().numpy()
    assert np.max(np.abs(rows - z["sisdr_rows0"])) <= 0.01, (rows, z["sisdr_rows0"])       # dB, north-star tolerance
    losses, _ = ops.sisdr_losses([est], b["wav_targets"])
    loss = losses[0]
    assert abs(float(loss.detach()) - float(z["loss"])) <= 2e-3
    loss.backward()
    worst = (0.0, "")
    for k, p in m.named_parameters():
        ref_n = float(z["gnorm/" + k])
        gn = float(p.grad.double().norm())
        rel = abs(gn - ref_n) / (ref_n + 1e-6)
        worst = max(worst, (rel, k))
        assert abs(gn - ref_n) <= tol_g * ref_n + 1e-5, (name, k, gn, ref_n)
        key = "g/" + k if "g/" + k in z else "ghead/" + k
        rg = torch.from_numpy(z[key]).to(DEV).reshape(-1).double()
        gg = p.grad.reshape(-1)[:rg.numel()].double()
        if float(rg.norm()) > 1e-6:
            cos = float((rg * gg).sum() / (rg.norm() * gg.norm() + 1e-30))
            assert cos >= 0.9995, (name, k, cos)
    print(name, "worst relative gradient-norm difference", worst)


def test_tfgridnet_golden_small():
    """2 blocks, 16 channels, hidden 32, 2 heads: 2 rows of 2089 samples; est, per-row SI-SDR, loss and every gradient."""
    _golden_case("tfgridnet_small_train")


def test_tfgridnet_golden_recipe_net():
    """tfgridnet.yaml network (6 blocks, 128 channels, hidden 192, 4 heads, qk 512) on 0.5 s: forward + SISDR + backward."""
    _golden_case("tfgridnet_full_train_05s")


def test_tfgridnet_golden_unfold_path():
    """emb_ks 4 / emb_hs 1 (the class default window): zero padding to whole windows, F.unfold, BLSTM over the windows,
    ConvTranspose1d as transposed product + overlap-add, crop; forward + SISDR + every gradient vs the real reference."""
    _golden_case("tfgridnet_small_ks4")


def test_tfgridnet_golden_packed_path():
    """emb_ks == emb_hs == 2: two positions per recurrent step (gridnet_block.py:139-146); vs the real reference."""
    _golden_case("tfgridnet_small_ks2")


@pytest.mark.parametrize("K,hs,T", [(4, 1, 71), (3, 2, 40), (4, 2, 10)])
def test_unfold_fold_1d(K, hs, T):
    """Unfold1dFn == F.unfold(x[..., None], (K, 1), stride=(hs, 1)); Fold1dFn == its adjoint (F.fold); both gradients."""
    import torch.nn.functional as F
    from wesep_b200 import ops
    n, C = 3, 8
    L = (T - K) // hs + 1
    x0 = rnd(n, C, T, seed=1)
    x = _act(x0)
    col = ops.Unfold1dFn.apply(x, K, hs)
    g0 = rnd(n, C * K, L, seed=2)
    col.backward(g0)
    x64 = x0.double().requires_grad_(True)
    ref = F.unfold(x64[..., None], (K, 1), stride=(hs, 1))
    ref.backward(g0.double())
    check("unfold", col.detach(), ref.detach(), 1e-7)
    check("unfold grad", x.grad, x64.grad, 1e-6)
    c = _act(g0)
    y = ops.Fold1dFn.apply(c, C, T, K, hs)
    gy = rnd(n, C, T, seed=3)
    y.backward(gy)
    c64 = g0.double().requires_grad_(True)
    ref2 = F.fold(c64, (T, 1), (K, 1), stride=(hs, 1))[..., 0]
    ref2.backward(gy.double())
    check("fold", y.detach(), ref2.detach(), 1e-6)
    check("fold grad", c.grad, c64.grad, 1e-7)
