"""Generate golden fixtures by running the REAL reference (/root/reference, imported in
place through oracle/stubs) on seeded inputs.  Run in the build container only:

    python tests/golden/make_golden.py

Weights and inputs are NOT stored: both sides regenerate them with
``wesep_b200.synth.fill_state_dict_(sd, seed)`` / ``make_batch(seed=...)`` (numpy PCG64,
machine independent).  Stored: reference outputs, loss parts, per-parameter gradient
norms (+ full gradients of small tensors); every fixture stays under 1 MB.  The reference ships no golden vectors
of its own (SURVEY.md §4), so these are the pin for oracle/*.py and, through it, for
the CUDA path.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import ref_loader, losses as olosses  # noqa: E402
from wesep_b200 import synth  # noqa: E402

SMALL = dict(B=64, H=128, X=3, R=2)


def grads_summary(model):
    out = {}
    for k, p in model.named_parameters():
        g = p.grad
        if g is None:
            continue
        g64 = g.double()
        out["gnorm/" + k] = np.float64(g64.norm().item())
        if g.numel() <= 4096:
            out["g/" + k] = g.detach().numpy().copy()
    return out


def run_case(get_model, name, args, n, T, Te, wseed, dseed, train=True, subsample=1, backward=True):
    torch.manual_seed(0)
    m = get_model("ConvTasNet")(**args)
    synth.fill_state_dict_(m.state_dict(), seed=wseed)
    b = synth.make_batch(n, T=T, Te=Te, seed=dseed)
    m.train(train)
    fix = {}
    with torch.set_grad_enabled(backward):
        out = m(b["wav_mix"], b["spk_embeds"])
        multi_task = args.get("multi_task", True)
        # T not a multiple of the hop: the decoder returns (K-1)*10+20 <= T samples; crop targets
        tgt = b["wav_targets"][:, :out[0].shape[-1]]
        loss, parts = olosses.train_loss(out, tgt, b["spk_label"], multi_task=multi_task)
    for i, o in enumerate(out):
        fix[f"out{i}"] = o.detach().numpy()[..., ::subsample].copy() if i < 3 else o.detach().numpy().copy()
    for i in range(3):
        fix[f"sisdr_rows{i}"] = olosses.sisdr_per_row(out[i].detach().double(), tgt.double()).numpy()
    fix["loss"] = np.float64(loss.item())
    for k, v in parts.items():
        fix["loss/" + k] = np.float64(v.item())
    if backward:
        loss.backward()
        fix.update(grads_summary(m))
    if train:
        for k, v in m.state_dict().items():
            if k.endswith("running_mean") or k.endswith("running_var"):
                fix["buf/" + k] = v.numpy().copy()
    meta = dict(name=name, args=args, n=n, T=T, Te=Te, wseed=wseed, dseed=dseed, train=train, subsample=subsample,
                backward=backward)
    fix["meta"] = np.array(json.dumps(meta))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **fix)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB", "loss", fix["loss"])


def run_optim():
    """3 steps of reference clip_gradients (wesep/utils/funcs.py:79-88) + torch.optim.Adam(wd=1e-4)."""
    from wesep.utils.funcs import clip_gradients

    class M(torch.nn.Module):
        def __init__(self, ps):
            super().__init__()
            self.ps = torch.nn.ParameterList(ps)

    rng = np.random.default_rng(11)
    shapes = [(7,), (33, 5), (1,), (64, 16, 3), (300,)]
    p0 = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    model = M([torch.nn.Parameter(torch.from_numpy(p.copy())) for p in p0])
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4)
    fix = {f"p0_{i}": p for i, p in enumerate(p0)}
    lrs = [1e-3, 9e-4, 5e-4]
    for step in range(3):
        for i, p in enumerate(model.ps):
            scale = [0.01, 3.0, 50.0, 0.2, 1.0][i]   # some tensors exceed clip=5, some don't
            g = (scale * rng.standard_normal(p.shape)).astype(np.float32)
            fix[f"g{step}_{i}"] = g
            p.grad = torch.from_numpy(g.copy())
        for gparam in opt.param_groups:
            gparam["lr"] = lrs[step]
        norms = clip_gradients(model, 5.0)
        fix[f"norms{step}"] = np.array(norms, np.float64)
        opt.step()
        for i, p in enumerate(model.ps):
            fix[f"p{step + 1}_{i}"] = p.detach().numpy().copy()
    fix["lrs"] = np.array(lrs)
    path = os.path.join(HERE, "optim.npz")
    np.savez_compressed(path, **fix)
    print("wrote", path)


def run_sched():
    from wesep.utils.schedulers import ExponentialDecrease
    opt = torch.optim.Adam([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
    s = ExponentialDecrease(opt, num_epochs=150, epoch_iter=1000, initial_lr=1e-3, final_lr=2.5e-5, warm_up_epoch=0,
                            warm_from_zero=False)
    its = [0, 1, 999, 75000, 149999]
    vals = []
    for it in its:
        s.step(it)
        vals.append(opt.param_groups[0]["lr"])
    np.savez(os.path.join(HERE, "sched.npz"), its=np.array(its), lrs=np.array(vals, np.float64))
    print("wrote sched", vals)


def run_sisnr():
    """In-tree numpy cal_SISNR formula (wesep/utils/score.py:7-21; the module itself needs pesq,
    so the 15 lines are exercised through oracle.losses.cal_sisnr_numpy which restates them)
    vs the restated auraloss SISDRLoss: fixture stores both for a range of SNRs."""
    rng = np.random.default_rng(7)
    rows = []
    for snr in (-30, -5, 0, 10, 40, 60):
        t = rng.standard_normal(64000).astype(np.float32) * 0.1 + 0.01
        e = rng.standard_normal(64000).astype(np.float32)
        e *= np.linalg.norm(t) / np.linalg.norm(e) * 10 ** (-snr / 20)
        x = (0.7 * t + e).astype(np.float32)
        a = float(olosses.sisdr_per_row(torch.from_numpy(x).double()[None], torch.from_numpy(t).double()[None])[0])
        c = float(olosses.cal_sisnr_numpy(t.astype(np.float64), x.astype(np.float64)))
        rows.append((snr, a, c))
    np.savez(os.path.join(HERE, "sisnr.npz"), rows=np.array(rows, np.float64))
    print("wrote sisnr", rows)


def main():
    ref_loader.import_reference()
    from wesep.models import get_model

    base = dict(ref_loader.SPEXPLUS_ARGS)
    small = dict(base)
    small.update(SMALL)
    # 1. small recipe-shaped config, train mode, fwd+bwd
    run_case(get_model, "spex_small_train", small, n=3, T=3200, Te=2400, wseed=3, dseed=5, train=True)
    run_case(get_model, "spex_small_eval", small, n=2, T=1999, Te=1503, wseed=4, dseed=6, train=False, backward=False)
    # n = 1 row (decoder.py:109-112 squeeze branch)
    run_case(get_model, "spex_small_n1", small, n=1, T=1600, Te=1600, wseed=8, dseed=9, train=False, backward=False)
    # 2. alternative fusion modes (separation.py:116-135)
    for ft in ("FiLM", "multiply", "additive", "concat"):
        a = dict(small)
        a.update(spk_fuse_type=ft)
        run_case(get_model, "spex_small_" + ft, a, n=2, T=1600, Te=1200, wseed=12, dseed=13, train=True)
    # 3. BASELINE config 1: full Spex+ on one 2-speaker mixture (n=2 rows), 4 s @ 16 kHz
    run_case(get_model, "spex_full_cfg1_eval", base, n=2, T=64000, Te=64000, wseed=0, dseed=1234, train=False,
             subsample=16, backward=False)
    run_case(get_model, "spex_full_cfg1_train", base, n=2, T=64000, Te=64000, wseed=0, dseed=1234, train=True,
             subsample=16, backward=True)
    run_optim()
    run_sched()
    run_sisnr()


if __name__ == "__main__":
    main()
