"""GPU: pDPCCN (SURVEY.md §8 row a23) — the streaming kernels of csrc/dpccn.cu and the im2col / col2im convolutions vs
fp64 torch restatements, and the whole model (forward, SISDR loss, every gradient) vs the golden outputs of the REAL
reference (tests/golden/dpccn_*.npz) and the fp64 oracle."""
import json
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import dpccn as od
from oracle import losses as olosses
from tests.test_gpu_kernels import check, rnd

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _act(t):
    from wesep_b200 import ops
    n, C = t.shape[:2]
    a = ops.new_act(n, C, t[0, 0].numel(), DEV)
    a.copy_(t.reshape(n, C, -1))
    return a.requires_grad_(True)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("L", [1503, 20000])
def test_elu_in(mode, L):
    from wesep_b200 import ops
    x0 = rnd(3, 5, L, seed=mode + L, scale=1.5)
    g0 = rnd(3, 5, L, seed=9)
    x = _act(x0)
    y = ops.EluInFn.apply(x, mode)
    y.backward(g0.to(DEV))
    x64 = x0.double().requires_grad_(True)
    r = od.inorm(od.elu(x64)) if mode == 0 else od.elu(od.inorm(x64))
    r.backward(g0.double())
    check("y", y.detach(), r.detach(), 2e-5)
    check("gx", x.grad, x64.grad, 5e-5)


@pytest.mark.parametrize("dil", [1, 4, 512])
def test_dwconv1d(dil):
    from wesep_b200 import ops
    n, C, L = 2, 12, 1503
    x0, w0, b0, g0 = rnd(n, C, L, seed=1), rnd(C, 1, 3, seed=2), rnd(C, seed=3), rnd(n, C, L, seed=4)
    x = _act(x0)
    w, b = w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    y = ops.DwConv1dFn.apply(x, w, b, dil)
    y.backward(g0.to(DEV))
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x0, w0, b0))
    r = F.conv1d(x64, w64, b64, padding=dil, dilation=dil, groups=C)
    r.backward(g0.double())
    check("y", y.detach(), r.detach(), 1e-5)
    check("gx", x.grad, x64.grad, 1e-5)
    check("gw", w.grad, w64.grad, 5e-5)
    check("gb", b.grad, b64.grad, 5e-5)


@pytest.mark.parametrize("k", [4, 32])
def test_avgpool_upsample(k):
    from wesep_b200 import ops
    n, C, H, W = 2, 3, 67, 129
    x0 = rnd(n, C, H, W, seed=k)
    x = _act(x0)
    p = ops.AvgPool2dFn.apply(x, H, W, k)
    u = ops.Upsample2dFn.apply(p, H // k, W // k, H, W)
    g0 = rnd(n, C, H * W, seed=5)
    u.backward(g0.to(DEV))
    x64 = x0.double().requires_grad_(True)
    p64 = F.avg_pool2d(x64, k)
    u64 = F.interpolate(p64, size=(H, W), mode="bilinear", align_corners=False)
    u64.backward(g0.double().reshape(n, C, H, W))
    check("pool", p.detach(), p64.detach().reshape(n, C, -1), 1e-5)
    check("up", u.detach(), u64.detach().reshape(n, C, -1), 1e-5)
    check("gx", x.grad, x64.grad.reshape(n, C, -1), 1e-5)


def test_colscale():
    from wesep_b200 import ops
    n, C, T, Fq = 2, 5, 33, 257
    x0, s0, g0 = rnd(n, C, T, Fq, seed=1), rnd(n, Fq, seed=2), rnd(n, C, T * Fq, seed=3)
    x = _act(x0)
    s = s0.clone().requires_grad_(True)
    y = ops.ColScaleFn.apply(x, s, T, Fq)
    y.backward(g0.to(DEV))
    x64, s64 = x0.double().requires_grad_(True), s0.double().requires_grad_(True)
    r = x64 * s64[:, None, None, :]
    r.backward(g0.double().reshape(n, C, T, Fq))
    check("y", y.detach(), r.detach().reshape(n, C, -1), 1e-6)
    check("gx", x.grad, x64.grad.reshape(n, C, -1), 1e-6)
    check("gs", s.grad, s64.grad, 2e-5)


@pytest.mark.parametrize("sw", [1, 2])
def test_conv3x3_stride_1x(sw):
    """Conv2d(3x3, padding 1, stride (1, sw)) = im2col + pointwise GEMM; forward and all gradients."""
    from wesep_b200 import ops
    n, Ci, Co, H, W = 2, 6, 8, 11, 33
    x0, w0, b0 = rnd(n, Ci, H, W, seed=1), rnd(Co, Ci, 3, 3, seed=2, scale=0.3), rnd(Co, seed=3)
    x = _act(x0)
    w, b = w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    y = ops.conv3x3(x, H, W, w, b, (1, sw))
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x0, w0, b0))
    r = F.conv2d(x64, w64, b64, stride=(1, sw), padding=(1, 1))
    g0 = rnd(*r.shape, seed=4)
    y.backward(g0.reshape(n, Co, -1).to(DEV))
    r.backward(g0.double())
    check("y", y.detach(), r.detach().reshape(n, Co, -1), 2e-5)
    check("gx", x.grad, x64.grad.reshape(n, Ci, -1), 2e-5)
    check("gw", w.grad, w64.grad, 5e-5)
    check("gb", b.grad, b64.grad, 5e-5)


@pytest.mark.parametrize("sw,Co", [(2, 8), (2, 2), (1, 2)])
def test_conv_transpose3x3(sw, Co):
    """ConvTranspose2d(3x3, padding 1, stride (1, sw)) = transposed pointwise GEMM + col2im (Co = 2: the padded product)."""
    from wesep_b200 import ops
    n, Ci, H, Wi = 2, 8, 9, 17
    x0, w0, b0 = rnd(n, Ci, H, Wi, seed=1), rnd(Ci, Co, 3, 3, seed=2, scale=0.3), rnd(Co, seed=3)
    x = _act(x0)
    w, b = w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    Wo = (Wi - 1) * sw + 1
    y = ops.conv_transpose3x3(x, H, Wo, w, b, (1, sw))
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x0, w0, b0))
    r = F.conv_transpose2d(x64, w64, b64, stride=(1, sw), padding=(1, 1))
    assert r.shape[-1] == Wo
    g0 = rnd(*r.shape, seed=4)
    y.backward(g0.reshape(n, Co, -1).to(DEV))
    r.backward(g0.double())
    check("y", y.detach(), r.detach().reshape(n, Co, -1), 2e-5)
    check("gx", x.grad, x64.grad.reshape(n, Ci, -1), 2e-5)
    check("gw", w.grad, w64.grad, 5e-5)
    check("gb", b.grad, b64.grad, 5e-5)


# the depthwise conv's bias feeds InstanceNorm directly (convs.py:146-148): a constant shift of a plane is removed by the
# norm, so its gradient is exactly 0 in exact arithmetic and both sides hold round-off only (|g| ~ 1e-7)
ZERO_GRAD = re.compile(r"tcn_layers\.\d+\.\d+\.dconv1\.bias$")


def _golden_case(name, tol_g=2e-3):
    from wesep_b200 import ops, synth
    from wesep_b200.models import get_model
    z = np.load(os.path.join(GOLD, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    m = get_model("DPCCN")(**meta["args"])
    ref_sd = od.make_state_dict(tcn_blocks=meta["args"]["tcn_blocks"], tcn_layers=meta["args"]["tcn_layers"])
    assert list(m.state_dict().keys()) == list(ref_sd.keys())
    synth.fill_state_dict_(m.state_dict(), seed=meta["wseed"])
    m = m.to(DEV).train()
    b = synth.make_batch(meta["n"], T=meta["L"], Te=8, seed=meta["dseed"], device=DEV)
    rng = np.random.default_rng(meta["dseed"] + 77)
    emb = torch.from_numpy(rng.standard_normal((meta["n"], 256)).astype(np.float32)).to(DEV)
    est, _ = m(b["wav_mix"], emb)
    ref = torch.from_numpy(z["out0"]).to(DEV)
    got = est.detach()[..., ::meta["subsample"]]
    assert got.shape == ref.shape
    check("est", got, ref, 5e-4)
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
        if ZERO_GRAD.search(k):
            assert gn <= 1e-4 and ref_n <= 1e-4, (name, k, gn, ref_n)
            continue
        rel = abs(gn - ref_n) / (ref_n + 1e-6)
        worst = max(worst, (rel, k))
        assert abs(gn - ref_n) <= tol_g * ref_n + 1e-5, (name, k, gn, ref_n)
        key ="g/" + k if "g/" + k in z else "ghead/" + k
        rg = torch.from_numpy(z[key]).to(DEV).reshape(-1).double()
        gg = p.grad.reshape(-1)[:rg.numel()].double()
        cos = float((rg * gg).sum() / (rg.norm() * gg.norm() + 1e-30))
        assert cos >= 0.9999, (name, k, cos)
    print(name, "worst relative gradient-norm difference", worst)


def test_dpccn_golden_small():
    """Reduced TCN depth (3 blocks x 1 layer), 2 rows of 4173 samples: est, per-row SI-SDR, loss and every gradient."""
    _golden_case("dpccn_small_train")


def test_dpccn_golden_recipe_net_1s():
    """dpccn.yaml network (10 blocks x 2 layers, 257 bins) on 1 s: forward + SISDR + backward vs the real reference."""
    _golden_case("dpccn_full_train_1s")


def test_dpccn_joint_training_constructs_and_steps():
    """dpccn.yaml model_args verbatim (joint ResNet34 on fbank features): constructs, one train step runs, every
    parameter receives a gradient (DDP requirement, train.py:63)."""
    from wesep_b200.models import get_model
    args = dict(win=512, stride=128, feature_dim=257, tcn_blocks=10, tcn_layers=2, causal=False, spk_fuse_type="multiply",
                use_spk_transform=False, multi_fuse=False, joint_training=True, spk_model="ResNet34", spk_model_init=False,
                spk_args=dict(feat_dim=80, embed_dim=256, pooling_func="TSTP", two_emb_layer=False), spk_emb_dim=256,
                spk_model_freeze=False, spk_feat=True, feat_type="consistent")
    m = get_model("DPCCN")(**args).to(DEV).train()
    g = torch.Generator().manual_seed(0)
    mix = (torch.randn(2, 8000, generator=g) * 0.1).to(DEV)
    fb = torch.randn(2, 60, 80, generator=g).to(DEV)
    est, emb = m(mix, fb)
    assert est.shape == (2, 8000) and emb.shape == (2, 256)
    est.square().mean().backward()
    missing = [k for k, p in m.named_parameters() if p.grad is None]
    assert not missing, missing
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())
