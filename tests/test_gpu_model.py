"""GPU parity of the whole Spex+ path against (a) golden outputs of the REAL reference
(tests/golden/*.npz) and (b) the oracle run in fp64, incl. the full train step."""
import numpy as np
import pytest
import torch

from oracle import losses as olosses
from oracle import optim as ooptim
from oracle import spexplus as ospex
from tests.util import ZERO_GRAD, cfg_from_args, fixture_inputs, load_fixture, rel_l2
from wesep_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"


def build_model(args, wseed):
    from wesep_b200.models import get_model
    m = get_model("ConvTasNet")(**args)
    synth.fill_state_dict_(m.state_dict(), seed=wseed)
    return m.to(DEV)


def run_fixture(name, check_grads=True):
    from wesep_b200.utils.executor import compute_loss
    z, meta = load_fixture(name)
    m = build_model(meta["args"], meta["wseed"])
    m.train(meta["train"])
    b = synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=meta["dseed"], device=DEV)
    with torch.set_grad_enabled(meta["backward"]):
        out = m(b["wav_mix"], b["spk_embeds"])
        loss, rows = compute_loss(out, b["wav_targets"], b["spk_label"], multi_task=meta["args"].get("multi_task", True))
    sub = meta["subsample"]
    report = {}
    for i in range(3):
        ref = torch.from_numpy(z[f"out{i}"]).to(DEV)
        got = out[i].detach()[..., ::sub]
        assert got.shape == ref.shape, (name, i, got.shape, ref.shape)
        report[f"out{i}"] = rel_l2(got, ref)
        assert report[f"out{i}"] <= 2e-4, (name, f"out{i}", report[f"out{i}"])
        d = float(np.max(np.abs(rows[i].detach().cpu().numpy() - z[f"sisdr_rows{i}"])))
        report[f"dB{i}"] = d
        assert d <= 0.01, (name, f"SI-SDR est{i + 1} differs by {d:.4f} dB (tolerance 0.01 dB)")
    if len(out) > 3:
        assert rel_l2(out[3].detach(), torch.from_numpy(z["out3"]).to(DEV)) <= 2e-4
    assert abs(float(loss) - float(z["loss"])) <= 1e-3 * abs(float(z["loss"])) + 2e-3, (float(loss), float(z["loss"]))
    if meta["backward"] and check_grads:
        # Gradients: the golden run is fp32 too; wherever a PReLU pre-activation is ~1e-7 the two fp32 runs may
        # take different branches (derivative jump), which moves isolated gradient elements by O(1) and, with only
        # K=319 frames in the small config, norms by up to ~1 %.  Arithmetic-level backward parity is pinned at
        # 3e-5 in tests/test_gpu_kernels.py with branch-pinned oracles; here we gate on norm + direction.
        loss.backward()
        tol_n, tol_g = (2e-2, 5e-2) if meta["T"] < 10000 else (1e-2, 2e-2)
        worst = 0.0
        for k, p in m.named_parameters():
            ref = float(z["gnorm/" + k])
            gn = float(p.grad.double().norm())
            if ZERO_GRAD.search(k):
                assert gn <= 1e-3 and ref <= 1e-3, (name, k, gn, ref)
                continue
            tn = 5e-2 if p.numel() <= 4 else tol_n     # scalar PReLU slopes: |sum of +/- terms|, fp32-noisy on both sides
            # scalar slopes: a sum of ~1e6 terms of either sign that cancels to ~2e-3; the two fp32 runs differ by up to
            # ~5e-4 there (measured 4.5e-4 on spk_model.aux_enc3.2.prelu1.weight at 4 s), hence the larger absolute floor
            floor = 1e-3 if p.numel() <= 4 else 3e-4
            assert abs(gn - ref) <= tn * ref + floor, (name, k, gn, ref)
            if ("g/" + k) in z and p.numel() > 4:
                g = torch.from_numpy(z["g/" + k]).to(DEV)
                e = float((p.grad - g).double().norm() / (g.double().norm() + 1e-3))
                worst = max(worst, e)
                assert e <= tol_g, (name, k, e)
        report["worst_small_grad_rel"] = worst
    if meta["train"]:
        for k, v in m.state_dict().items():
            if k.endswith("running_mean") or k.endswith("running_var"):
                assert torch.allclose(v.cpu(), torch.from_numpy(z["buf/" + k]), rtol=1e-3, atol=1e-5), (name, k)
    return report


@pytest.mark.parametrize("name", ["spex_small_train", "spex_small_eval", "spex_small_n1"])
def test_golden_small(name):
    run_fixture(name)


@pytest.mark.parametrize("ft", ["FiLM", "multiply", "additive", "concat"])
def test_golden_alternative_fusion(ft):
    """spk_fuse_type variants of FuseSeparation (separation.py:116-135) vs goldens of the real reference."""
    run_fixture("spex_small_" + ft)


def test_golden_full_cfg1_eval():
    """BASELINE config 1: Spex+ forward + SI-SNR, one 2-speaker 4 s mixture, vs the real reference."""
    run_fixture("spex_full_cfg1_eval")


def test_golden_full_cfg1_train():
    run_fixture("spex_full_cfg1_train")


def test_full_model_vs_oracle_fp64_all_grads():
    """Every output and EVERY parameter gradient of the small config vs the fp64 oracle."""
    from wesep_b200.utils.executor import compute_loss
    z, meta = load_fixture("spex_small_train")
    m = build_model(meta["args"], meta["wseed"])
    m.train()
    b = synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=meta["dseed"], device=DEV)
    out = m(b["wav_mix"], b["spk_embeds"])
    loss, _ = compute_loss(out, b["wav_targets"], b["spk_label"])
    loss.backward()
    cfg, sd, _ = fixture_inputs(meta, dtype=torch.float64, device=DEV)
    names = [k for k, _ in m.named_parameters()]
    for k in names:
        sd[k].requires_grad_(True)
    o64 = ospex.convtasnet_forward(sd, cfg, b["wav_mix"].double(), b["spk_embeds"].double(), training=True)
    l64, _ = olosses.train_loss(o64, b["wav_targets"].double(), b["spk_label"])
    l64.backward()
    assert abs(float(loss) - float(l64)) <= 2e-3
    for i in range(4):
        assert rel_l2(out[i].detach(), o64[i].detach()) <= 5e-5, i
    bad = []
    for k, p in m.named_parameters():
        if ZERO_GRAD.search(k):
            assert float(p.grad.abs().max()) <= 1e-3
            continue
        e = float((p.grad.double() - sd[k].grad).norm() / (sd[k].grad.norm() + 1e-3))
        if e > 3e-2:          # PReLU-kink branch flips (see run_fixture) bound this comparison, not the arithmetic
            bad.append((k, e))
    assert not bad, bad[:10]


def test_train_steps_vs_oracle():
    """3 full train steps (fwd, loss, bwd, per-tensor clip, Adam wd=1e-4, exp-decay lr) vs the oracle loop."""
    from wesep_b200.utils.executor import train_step
    from wesep_b200.utils.optim import FusedClipAdam
    z, meta = load_fixture("spex_small_train")
    m = build_model(meta["args"], meta["wseed"])
    m.train()
    opt = FusedClipAdam(m.parameters(), lr=1e-3, weight_decay=1e-4, clip=5.0)
    cfg, sd, _ = fixture_inputs(meta, dtype=torch.float64, device=DEV)
    names = [k for k, _ in m.named_parameters()]
    P = [sd[k].requires_grad_(True) for k in names]
    mom = [torch.zeros_like(p) for p in P]
    var = [torch.zeros_like(p) for p in P]
    losses, ref_losses = [], []
    for step in range(3):
        lr = ooptim.exponential_decrease_lr(step, 1000)
        b = synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=100 + step, device=DEV)
        opt.param_groups[0]["lr"] = lr
        losses.append(float(train_step(m, b, opt)))
        bufs = {}
        o64 = ospex.convtasnet_forward(sd, cfg, b["wav_mix"].double(), b["spk_embeds"].double(), training=True,
                                       buffers_out=bufs)
        l64, _ = olosses.train_loss(o64, b["wav_targets"].double(), b["spk_label"])
        grads = torch.autograd.grad(l64, P)
        grads = [g.clone() for g in grads]
        ooptim.clip_gradients(grads, 5.0)
        with torch.no_grad():
            ooptim.adam_step(P, grads, mom, var, step + 1, lr)
            sd.update(bufs)
        ref_losses.append(float(l64))
    assert np.allclose(losses, ref_losses, rtol=2e-3, atol=2e-3), (losses, ref_losses)
    # Adam's first steps move every element by ~lr*sign(g), so any element whose gradient is below the fp32 /
    # branch-flip noise may move the other way (the fused clip+Adam arithmetic itself is checked exactly in
    # test_gpu_kernels.py::test_clip_adam_*).  Gate on the loss trajectory (above) and on >= 85 % of all
    # parameter elements agreeing with the fp64 oracle trajectory to 2e-4 after 3 steps.
    tot = bad = 0
    per = []
    for k, p in m.named_parameters():
        d = (p.detach().double() - sd[k].detach()).abs()
        tot += d.numel()
        b_ = int((d > 2e-4).sum())
        bad += b_
        if b_:
            per.append((b_ / d.numel(), b_, k))
    per.sort(reverse=True)
    assert bad <= 0.15 * tot, (bad, tot, per[:8])


def test_cuda_graph_train_step_matches_eager():
    """GraphedTrainStep (whole step captured once, replayed) vs the eager train_step: same batches, a moving learning rate,
    identical loss trajectory and parameters (the only difference is fp32 atomics ordering, already present run to run)."""
    from wesep_b200.utils.executor import GraphedTrainStep, train_step
    from wesep_b200.utils.optim import FusedClipAdam
    _, meta = load_fixture("spex_small_train")
    batches = [synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=200 + i, device=DEV) for i in range(6)]
    lrs = [ooptim.exponential_decrease_lr(i, 50) for i in range(6)]

    def run(graph):
        m = build_model(meta["args"], meta["wseed"])
        m.train()
        opt = FusedClipAdam(m.parameters(), lr=1e-3, weight_decay=1e-4, clip=5.0)
        p0 = opt.arena.flat_p.clone()
        losses = []
        if graph:
            # the constructor warms up with real optimizer steps on the example batch but must RESTORE parameters, Adam
            # state, step count and BatchNorm buffers afterwards: training starts from the state it was given
            step = GraphedTrainStep(m, opt, batches[0], warmup=2)
            assert opt.step_count == 0 and torch.equal(opt.arena.flat_p, p0)
            assert float(opt.exp_avg.abs().max()) == 0.0 and float(opt.exp_avg_sq.abs().max()) == 0.0
            for k, b in m.named_buffers():
                if k.endswith("num_batches_tracked"):
                    assert int(b) == 0, k
            for i in range(6):
                opt.param_groups[0]["lr"] = lrs[i]
                losses.append(float(step(batches[i])))
        else:
            for i in range(6):
                opt.param_groups[0]["lr"] = lrs[i]
                losses.append(float(train_step(m, batches[i], opt)))
        return losses, {k: p.detach().clone() for k, p in m.named_parameters()}, opt.step_count

    le, pe, se = run(False)
    lg, pg, sg = run(True)
    assert se == sg == 6
    assert np.allclose(lg, le, rtol=1e-3, atol=1e-3), (lg, le)
    # parameters: skip the decoder biases (their gradient is pure round-off, see ZERO_GRAD: Adam then moves them by
    # +-lr per step in a direction that depends on the order of fp32 atomics).  Two fp32 runs differ by 1.0e-3 .. 1.6e-3
    # in relative L2 after 6 Adam steps (measured over repeated runs: elements whose gradient is at the atomics-order
    # noise level move +-lr either way); a wrong schedule / stale scalar in the graph would show as >= 1e-2.
    num = sum(float((pg[k].double() - pe[k].double()).pow(2).sum()) for k in pe if not ZERO_GRAD.search(k))
    den = sum(float(pe[k].double().pow(2).sum()) for k in pe if not ZERO_GRAD.search(k))
    assert (num / den) ** 0.5 < 3e-3, (num / den) ** 0.5
