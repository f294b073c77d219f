"""GPU: pBSRNN building blocks (SURVEY.md §8 rows a19-a20) vs the fp64 oracle (oracle/bsrnn.py): layout swap, LSTM cell,
the time-major BLSTM Function, ResRNN and BSNet, forward and all gradients."""
import pytest
import torch

from oracle import bsrnn as ob
from tests.test_gpu_kernels import check, rnd

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("nb,Q,C,S", [(1, 5, 3, 70), (2, 32, 16, 33), (3, 40, 4, 7)])
def test_swap_outer_inner(nb, Q, C, S):
    from wesep_b200 import ops
    x = ops.new_act(nb * Q, C, S, DEV)
    x.copy_(rnd(nb * Q, C, S, seed=1))
    res = ops.new_act(nb * S, C, Q, DEV)
    res.copy_(rnd(nb * S, C, Q, seed=2))
    xr = x.detach().clone().requires_grad_(True)
    rr = res.detach().clone().requires_grad_(True)
    y = ops.SwapOIFn.apply(xr, nb, rr)
    ref = x.view(nb, Q, C, S).permute(0, 3, 2, 1).reshape(nb * S, C, Q) + res
    assert torch.equal(y, ref)
    g = rnd(nb * S, C, Q, seed=3)
    y.backward(g)
    assert torch.equal(xr.grad, g.view(nb, S, C, Q).permute(0, 3, 2, 1).reshape(nb * Q, C, S))
    assert torch.equal(rr.grad, g)
    assert torch.equal(ops.SwapOIFn.apply(x, nb, None), x.view(nb, Q, C, S).permute(0, 3, 2, 1).reshape(nb * S, C, Q))


def _lstm_params(C, Hd, seed):
    ps = []
    for d in range(2):
        ps += [rnd(4 * Hd, C, seed=seed + 10 * d, scale=C ** -0.5), rnd(4 * Hd, Hd, seed=seed + 10 * d + 1, scale=Hd ** -0.5),
               rnd(4 * Hd, seed=seed + 10 * d + 2, scale=0.1), rnd(4 * Hd, seed=seed + 10 * d + 3, scale=0.1)]
    return ps


@pytest.mark.parametrize("Q,C,S,Hd", [(6, 16, 9, 32), (70, 32, 5, 64), (33, 128, 12, 256)])
def test_blstm_time_major(Q, C, S, Hd):
    """LstmTmFn vs the explicit recurrence of the oracle (lstm_dir), forward and every gradient."""
    from wesep_b200 import ops
    xs = rnd(Q, S, C, seed=1)                                  # oracle layout [N, S, I]
    ps = _lstm_params(C, Hd, 5)
    xn = ops.new_act(S, C, Q, DEV)
    xn.copy_(xs.permute(1, 2, 0))
    xn.requires_grad_(True)
    pg = [p.clone().requires_grad_(True) for p in ps]
    h = ops.LstmTmFn.apply(xn, *pg)
    x64 = xs.double().requires_grad_(True)
    p64 = [p.double().requires_grad_(True) for p in ps]
    hf = ob.lstm_dir(x64, *p64[:4], False)
    hb = ob.lstm_dir(x64, *p64[4:], True)
    ref = torch.cat([hf, hb], 2).permute(1, 2, 0)              # [S, 2Hd, Q]
    check("h", h, ref, 2e-5)
    g = rnd(S, 2 * Hd, Q, seed=9)
    h.backward(g)
    ref.backward(g.double())
    check("dx", xn.grad, x64.grad.permute(1, 2, 0), 1e-4)
    for name, a, b in zip(["w_ih", "w_hh", "b_ih", "b_hh"] * 2, pg, p64):
        check(name, a.grad, b.grad, 2e-4)


@pytest.mark.parametrize("Q,C,S", [(6, 16, 40), (64, 128, 20)])
def test_res_rnn(Q, C, S):
    from wesep_b200 import ops
    Hd = 2 * C
    sd = {"norm.weight": 1 + 0.1 * rnd(C, seed=1), "norm.bias": 0.1 * rnd(C, seed=2),
          "proj.weight": rnd(C, 2 * Hd, seed=3, scale=(2 * Hd) ** -0.5), "proj.bias": 0.1 * rnd(C, seed=4)}
    lp = _lstm_params(C, Hd, 20)
    for k, v in zip(["rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0", "rnn.bias_hh_l0", "rnn.weight_ih_l0_reverse",
                     "rnn.weight_hh_l0_reverse", "rnn.bias_ih_l0_reverse", "rnn.bias_hh_l0_reverse"], lp):
        sd[k] = v
    x0 = rnd(Q, C, S, seed=7)
    x = ops.new_act(Q, C, S, DEV)
    x.copy_(x0)
    x.requires_grad_(True)
    P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    y = ops.res_rnn(x, P["norm.weight"], P["norm.bias"], [P[k] for k in list(sd)[4:]], P["proj.weight"], P["proj.bias"])
    x64 = x0.double().requires_grad_(True)
    P64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    ref = ob.res_rnn(x64, P64, "")
    check("y", y, ref, 2e-5)
    g = rnd(Q, C, S, seed=8)
    y.backward(g)
    ref.backward(g.double())
    check("dx", x.grad, x64.grad, 2e-4)
    for k in sd:
        check(k, P[k].grad, P64[k].grad, 5e-4)


def test_bsnet_vs_oracle():
    """BSNet (band_rnn over time, permute, band_comm over bands, permute back) vs oracle.bsnet, forward + input gradient."""
    from wesep_b200 import ops, synth
    from wesep_b200.models.bsrnn import BSNet
    B, nb, N, T = 2, 5, 16, 21
    net = BSNet(nb * N, nb)
    synth.fill_state_dict_(net.state_dict(), seed=4)
    net = net.to(DEV)
    x0 = rnd(B, nb * N, T, seed=2)
    x = ops.new_act(B, nb * N, T, DEV)
    x.copy_(x0)
    x.requires_grad_(True)

    def args(m):
        r = m.rnn
        return (m.norm.weight, m.norm.bias, [r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, r.weight_ih_l0_reverse,
                                             r.weight_hh_l0_reverse, r.bias_ih_l0_reverse, r.bias_hh_l0_reverse],
                m.proj.weight, m.proj.bias)
    y = ops.bsnet(x, nb, args(net.band_rnn), args(net.band_comm))
    sd = {k: v.detach().double() for k, v in net.state_dict().items()}
    x64 = x0.double().requires_grad_(True)
    ref = ob.bsnet(x64, sd, "", nb)
    check("y", y, ref, 5e-5)
    g = rnd(B, nb * N, T, seed=3)
    y.backward(g)
    ref.backward(g.double())
    check("dx", x.grad, x64.grad, 5e-4)


def _golden_case(name, backward, tol=dict(gnorm=5e-4, g=5e-4, cos=0.9999)):   # measured on B200: <= 7.5e-5, 7.6e-5, 1 - 1e-10
    import json, os
    import numpy as np
    from oracle import losses as olosses
    from wesep_b200 import ops, synth
    from wesep_b200.models import get_model
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    m = get_model("BSRNN")(**meta["args"])
    synth.fill_state_dict_(m.state_dict(), seed=meta["wseed"])
    m = m.to(DEV).train()
    b = synth.make_batch(meta["n"], T=meta["L"], Te=8, seed=meta["dseed"], device=DEV)
    rng = np.random.default_rng(meta["dseed"] + 77)
    emb = torch.from_numpy(rng.standard_normal((meta["n"], 256)).astype(np.float32)).to(DEV)
    est, _ = m(b["wav_mix"], emb)
    ref = torch.from_numpy(z["out0"]).to(DEV)
    got = est.detach()[..., ::meta["subsample"]]
    assert got.shape == ref.shape
    check("est", got, ref, 2e-3)
    rows = olosses.sisdr_per_row(est.detach().double(), b["wav_targets"].double()).cpu().numpy()
    assert np.max(np.abs(rows - z["sisdr_rows0"])) <= 0.01, (rows, z["sisdr_rows0"])       # dB, north-star tolerance
    if backward:
        losses, _ = ops.sisdr_losses([est], b["wav_targets"])
        loss = losses[0]
        assert abs(float(loss) - float(z["loss"])) <= 2e-3, (float(loss), float(z["loss"]))
        loss.backward()
        bad, worst = [], dict(gnorm=0.0, g=0.0, cos=1.0)
        tot = sum(float(z[k]) ** 2 for k in z.files if k.startswith("gnorm/")) ** 0.5
        for k, p in m.named_parameters():
            ref_n = float(z["gnorm/" + k])
            g = p.grad.double()
            gn = float(g.norm())
            rel = abs(gn - ref_n) / (ref_n + 1e-12)
            if ref_n > 1e-6 * tot:                       # tensors whose gradient is not round-off
                worst["gnorm"] = max(worst["gnorm"], rel)
                if rel > tol["gnorm"]:
                    bad.append(("gnorm", k, gn, ref_n))
                if "g/" + k in z.files:                  # full gradient of the small tensors
                    r = torch.from_numpy(z["g/" + k]).to(DEV).double()
                    e = float((g - r).norm() / (r.norm() + 1e-30))
                    worst["g"] = max(worst["g"], e)
                    if e > tol["g"]:
                        bad.append(("g", k, e))
                if "ghead/" + k in z.files:              # direction of the large ones (first 256 elements)
                    r = torch.from_numpy(z["ghead/" + k]).to(DEV).double()
                    h = g.reshape(-1)[:256]
                    if float(r.norm()) > 1e-6 * tot:
                        c = float((h * r).sum() / (h.norm() * r.norm() + 1e-30))
                        worst["cos"] = min(worst["cos"], c)
                        if c < tol["cos"]:
                            bad.append(("cos", k, c))
        print(name, "worst gradient differences", worst)
        assert not bad, (worst, bad[:8])


@pytest.mark.parametrize("name", ["bsrnn_small_multiply", "bsrnn_small_additive_multi", "bsrnn_small_concat"])
def test_bsrnn_golden_small(name):
    """Whole pBSRNN (STFT -> band split -> fuse -> 2 x BSNet -> mask head -> iSTFT) + SISDR loss + backward vs golden
    outputs / loss / gradient norms of the real reference."""
    _golden_case(name, backward=True)


def test_bsrnn_golden_recipe_size_train_4s():
    """BASELINE config 3 as benchmarked: bsrnn.yaml-size network, 4 s, 2 rows — estimate, per-row SI-SDR within 0.01 dB, loss,
    every gradient norm, the full gradient of every small tensor and the direction of the large ones vs the real reference."""
    _golden_case("bsrnn_full_train_4s", backward=True)


def test_bsrnn_golden_recipe_size_forward():
    """bsrnn.yaml network (feature 128, hidden 256, 6 repeats, 32 bands) on 1 s of audio vs the reference, forward."""
    _golden_case("bsrnn_full_fwd_1s", backward=False)


@pytest.mark.parametrize("seqs", [0, 64, 128])
@pytest.mark.parametrize("Q,C,S,Hd", [(5, 16, 3, 32), (64, 32, 7, 64), (100, 16, 6, 128), (70, 24, 5, 192), (130, 128, 33, 256),
                                      (512, 128, 9, 256)])
def test_lstm_rec_matches_step_loop(Q, C, S, Hd, seqs, monkeypatch):
    """The persistent cluster recurrence (wesep_b200_lstm_rec_fwd / _bwd) vs the step-by-step path (one fp32-grade GEMM +
    one cell kernel per step) on the same inputs: h, dx and every parameter gradient."""
    from wesep_b200 import ops
    xs = rnd(S, C, Q, seed=1)
    ps = _lstm_params(C, Hd, 5)
    g = rnd(S, 2 * Hd, Q, seed=9)
    outs = []
    monkeypatch.setenv("WESEP_LSTM_REC_SEQS", str(seqs))
    for flag in ("0", "1"):
        monkeypatch.setenv("WESEP_LSTM_REC", flag)
        xn = ops.new_act(S, C, Q, DEV)
        xn.copy_(xs)
        xn.requires_grad_(True)
        pg = [p.clone().requires_grad_(True) for p in ps]
        h = ops.LstmTmFn.apply(xn, *pg)
        h.backward(g)
        outs.append([h.detach(), xn.grad] + [p.grad for p in pg])
    names = ["h", "dx"] + ["w_ih", "w_hh", "b_ih", "b_hh"] * 2
    for nm, a, b in zip(names, *outs):
        check(nm, b, a.double(), 2e-5 if nm == "h" else 1e-4)


def test_lstm_second_backward_raises():
    from wesep_b200 import ops
    xn = ops.new_act(3, 8, 4, DEV)
    xn.copy_(rnd(3, 8, 4, seed=1))
    xn.requires_grad_(True)
    h = ops.LstmTmFn.apply(xn, *[p.requires_grad_(True) for p in _lstm_params(8, 32, 5)])
    h.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        h.sum().backward()


@pytest.mark.parametrize("n,C,T,sliced", [(5, 6, 501, False), (70, 16, 32, False), (3, 128, 501, True), (9, 32, 37, True),
                                            (2, 16, 40003, False), (2, 8, 70001, True)])   # the last two: wide rows (>= 2^19 elements)
def test_group_norm1(n, C, T, sliced):
    """GroupNorm(1, C) one-CTA-per-row kernels vs torch.nn.functional.group_norm in fp64 (forward, dx, dgamma, dbeta);
    `sliced`: the input is a channel slice of a larger act tensor (batch stride > C * ld)."""
    import torch.nn.functional as F
    from wesep_b200 import ops
    Cbig = C + 8 if sliced else C
    xb = ops.new_act(n, Cbig, T, DEV)
    xb.copy_(rnd(n, Cbig, T, seed=1) * 3.0 + 0.5)
    x0 = xb[:, 4:4 + C] if sliced else xb
    w0, b0 = 1 + 0.2 * rnd(C, seed=2), 0.3 * rnd(C, seed=3)
    x = x0.detach().requires_grad_(True)
    w, b = w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    y = ops.group_norm1(x, w, b)
    x64 = x0.detach().double().contiguous().requires_grad_(True)
    w64, b64 = w0.double().requires_grad_(True), b0.double().requires_grad_(True)
    ref = F.group_norm(x64, 1, w64, b64, ops.GN_EPS)
    check("y", y, ref, 2e-6)
    g = rnd(n, C, T, seed=4)
    y.backward(g)
    ref.backward(g.double())
    check("dx", x.grad, x64.grad, 2e-5)
    check("dgamma", w.grad, w64.grad, 2e-5)
    check("dbeta", b.grad, b64.grad, 2e-5)


def test_bsrnn_multi_golden():
    """BSRNN_Multi (SURVEY 8f-4; bsrnn_multi_optim.py:406-472): first and self-enrolled second estimate, the weighted loss of
    the recipe (0.4 / 0.6) and every gradient vs the REAL reference run (tests/golden/bsrnn_multi_small.npz); under no_grad
    the model returns the two-tuple of the first pass.  Raw-wave enrollment -> "consistent" features inside the model."""
    import json, os
    import numpy as np
    from oracle import losses as olosses
    from tests.util import SqTiny
    from wesep_b200 import ops, synth
    from wesep_b200.models import get_model
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bsrnn_multi_small.npz"))
    meta = json.loads(str(z["meta"]))
    m = get_model("BSRNN_Multi")(**dict(meta["args"], spk_args=dict(feat_dim=80, embed_dim=256, pooling_func="TSTP",
                                                                      two_emb_layer=False)))
    m.spk_model = SqTiny(80, 256)                       # the stand-in the golden run used (wespeaker is external)
    params = {k: v for k, v in m.state_dict().items() if not k.startswith(("preEmphasis", "spk_encoder"))}
    synth.fill_state_dict_(params, seed=meta["wseed"])
    m = m.to(DEV).train()
    b = synth.make_batch(meta["n"], T=meta["L"], Te=meta["Te"], seed=meta["dseed"], device=DEV)
    out = m(b["wav_mix"], b["spk_embeds"])
    assert len(out) == 4
    s, self_s = out[0], out[1]
    for i, est in enumerate((s, self_s)):
        check(f"out{i}", est.detach(), torch.from_numpy(z[f"out{i}"]).to(DEV), 2e-3)
        rows = olosses.sisdr_per_row(est.detach().double(), b["wav_targets"].double()).cpu().numpy()
        assert np.max(np.abs(rows - z[f"sisdr_rows{i}"])) <= 0.01, (i, rows, z[f"sisdr_rows{i}"])
    losses, _ = ops.sisdr_losses([s, self_s], b["wav_targets"])
    loss = 0.4 * losses[0] + 0.6 * losses[1]
    assert abs(float(loss.detach()) - float(z["loss"])) <= 2e-3
    loss.backward()
    for k, p in m.named_parameters():
        ref_n, gn = float(z["gnorm/" + k]), float(p.grad.double().norm())
        assert abs(gn - ref_n) <= 2e-3 * ref_n + 1e-5, (k, gn, ref_n)
        rg = torch.from_numpy(z["ghead/" + k]).to(DEV).reshape(-1).double()
        gg = p.grad.reshape(-1)[:rg.numel()].double()
        if float(rg.norm()) > 1e-6:
            assert float((rg * gg).sum() / (rg.norm() * gg.norm() + 1e-30)) >= 0.9995, k
    m.eval()
    with torch.no_grad():
        out = m(b["wav_mix"], b["spk_embeds"])
    assert len(out) == 2
    check("eval", out[0], torch.from_numpy(z["eval_out0"]).to(DEV), 2e-3)
