"""Golden fixtures that pin the oracle to the REAL reference modules (imported in place through oracle/stubs) without
needing the reference at test time.  Run in the build container only:

    python tests/golden/make_golden_layouts.py

Writes
  state_dict_layouts.npz    `layouts`: JSON of the [key, shape] lists, in order, of the reference ConvTasNet (small config,
                            three fusion types) and BSRNN (joint_training False, two fusion settings) state_dicts
  spex_small_sumsq.npz      reference ConvTasNet (small config, train mode) in fp64 on seeded weights / inputs: the norm of
                            each of the four outputs and its elements at ``sample_index(numel, OUT_SAMPLE)``; for the loss
                            sum of squares of the outputs, every gradient's norm (`gnorm`) and its elements at
                            ``sample_index(numel, GRAD_SAMPLE)`` (`gsample`), concatenated in the order of meta["params"].  fp64 so that the comparison does not depend on the
                            reduction order of the CPU that runs it; samples plus full norms keep the fixture small.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import ref_loader  # noqa: E402
from wesep_b200 import synth  # noqa: E402

SMALL = dict(B=64, H=128, X=3, R=2)
SPEX_FUSE_TYPES = ("concatConv", "FiLM", "multiply")
BSRNN_BASE = dict(spk_emb_dim=256, sr=16000, win=512, stride=128, feature_dim=16, num_repeat=2, use_spk_transform=False,
                  joint_training=False)
BSRNN_FUSE = (("multiply", False), ("concat", True))
OUT_SAMPLE = 512
GRAD_SAMPLE = 64


def sample_index(numel, cap):
    """Evenly strided element indices, at most `cap` of them (tests/test_oracle_vs_reference.py repeats the rule)."""
    return np.arange(0, numel, -(-numel // cap))


def layouts():
    from wesep.models import get_model
    from wesep.models.bsrnn import BSRNN
    out = {}
    for ft in SPEX_FUSE_TYPES:
        args = dict(ref_loader.SPEXPLUS_ARGS, spk_fuse_type=ft, **SMALL)
        out["spex/" + ft] = [[k, list(v.shape)] for k, v in get_model("ConvTasNet")(**args).state_dict().items()]
    for fuse, mf in BSRNN_FUSE:
        m = BSRNN(**dict(BSRNN_BASE, spk_fuse_type=fuse, multi_fuse=mf))
        out[f"bsrnn/{fuse}/multi_fuse={mf}"] = [[k, list(v.shape)] for k, v in m.state_dict().items()]
    path = os.path.join(HERE, "state_dict_layouts.npz")
    np.savez_compressed(path, layouts=np.array(json.dumps(out)))
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def spex_sumsq(n=2, T=2400, Te=1800, wseed=21, dseed=22):
    from wesep.models import get_model
    args = dict(ref_loader.SPEXPLUS_ARGS, **SMALL)
    torch.manual_seed(0)
    m = get_model("ConvTasNet")(**args).double()
    synth.fill_state_dict_(m.state_dict(), seed=wseed)
    b = synth.make_batch(n, T=T, Te=Te, seed=dseed, dtype=torch.float64)
    m.train()
    out = m(b["wav_mix"], b["spk_embeds"])
    fix = {}
    for i, o in enumerate(out):
        o = o.detach().reshape(-1)
        fix[f"onorm{i}"] = np.float64(o.norm().item())
        fix[f"osample{i}"] = o.numpy()[sample_index(o.numel(), OUT_SAMPLE)].copy()
    sum(o.square().sum() for o in out).backward()
    params = [k for k, _ in m.named_parameters()]
    grads = [p.grad.detach().reshape(-1).numpy() for _, p in m.named_parameters()]
    fix["gnorm"] = np.array([np.linalg.norm(g) for g in grads])
    fix["gsample"] = np.concatenate([g[sample_index(g.size, GRAD_SAMPLE)] for g in grads])
    meta = dict(args=args, n=n, T=T, Te=Te, wseed=wseed, dseed=dseed, out_sample=OUT_SAMPLE, grad_sample=GRAD_SAMPLE,
                params=params)
    fix["meta"] = np.array(json.dumps(meta))
    path = os.path.join(HERE, "spex_small_sumsq.npz")
    np.savez_compressed(path, **fix)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main():
    ref_loader.import_reference()
    layouts()
    spex_sumsq()


if __name__ == "__main__":
    main()
