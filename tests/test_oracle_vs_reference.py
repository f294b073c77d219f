"""CPU: oracle restatement vs the REAL reference modules, through fixtures of their runs
(tests/golden/state_dict_layouts.npz, tests/golden/spex_small_sumsq.npz; tests/golden/make_golden_layouts.py)."""
import pytest
import torch

from oracle import spexplus as ospex
from tests.util import load_fixture, load_layouts
from wesep_b200 import synth


def _sample_index(numel, cap):
    """The element sample the fixture stores: evenly strided, at most `cap` indices (make_golden_layouts.sample_index)."""
    return torch.arange(0, numel, -(-numel // cap))


@pytest.mark.parametrize("ft", ["concatConv", "FiLM", "multiply"])
def test_state_dict_contract(ft):
    ref = [(k, tuple(s)) for k, s in load_layouts()["spex/" + ft]]
    cfg = dict(ospex.DEFAULT_CFG)
    cfg.update(B=64, H=128, X=3, R=2, spk_fuse_type=ft)
    assert ref == ospex.state_dict_spec(cfg)


def test_forward_backward_matches_reference():
    """Both sides in fp64 (the fixture is a fp64 run of the reference), so the tolerances hold on any CPU.  Every output and
    gradient is checked through its norm and a strided sample of its elements."""
    z, meta = load_fixture("spex_small_sumsq")
    cfg = dict(ospex.DEFAULT_CFG)
    cfg.update(B=64, H=128, X=3, R=2)
    sd = ospex.make_state_dict(cfg, dtype=torch.float64)
    synth.fill_state_dict_(sd, seed=meta["wseed"])
    params = meta["params"]
    assert params == [k for k, v in sd.items() if v.is_floating_point() and "running_" not in k]
    for k in params:
        sd[k].requires_grad_(True)
    b = synth.make_batch(meta["n"], T=meta["T"], Te=meta["Te"], seed=meta["dseed"], dtype=torch.float64)
    out_o = ospex.convtasnet_forward(sd, cfg, b["wav_mix"], b["spk_embeds"], training=True)
    assert len(out_o) == sum(f.startswith("onorm") for f in z.files)
    for i, c in enumerate(out_o):
        c = c.detach().reshape(-1)
        assert abs(float(c.norm()) - float(z[f"onorm{i}"])) <= 1e-5 * float(z[f"onorm{i}"]) + 1e-6, i
        a = torch.from_numpy(z[f"osample{i}"])
        got = c[_sample_index(c.numel(), meta["out_sample"])]
        assert torch.allclose(a, got, rtol=1e-5, atol=1e-6), (i, float((a - got).abs().max()))
    sum(o.square().sum() for o in out_o).backward()
    gsample, off = torch.from_numpy(z["gsample"]), 0
    for k, ref_n in zip(params, z["gnorm"]):
        g = sd[k].grad.reshape(-1)
        assert abs(float(g.norm()) - float(ref_n)) <= 1e-4 * float(ref_n) + 1e-6, k
        got = g[_sample_index(g.numel(), meta["grad_sample"])]
        ref = gsample[off:off + got.numel()]
        off += got.numel()
        assert torch.allclose(ref, got, rtol=1e-4, atol=1e-6), k
    assert off == gsample.numel()
