#!/usr/bin/env python
"""bench.py — train-step throughput (utterances/sec) on synthetic 4 s @ 16 kHz two-speaker mixtures.

Headline (BASELINE.json `metric`, configs[1]; configs[3] for N > 1): Spex+, 32 model rows per GPU.
Second block `pbsrnn` (the other model the metric's target names; configs[2]): pBSRNN, bsrnn.yaml network, 16 rows per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows 32] [--bsrnn-rows 16]
                  [--dump-outputs DIR]

A "step" = forward + loss (Spex+: 0.8/0.1/0.1 SI-SDR + 0.5 CE; pBSRNN: SI-SDR) + backward + gradient all-reduce (N > 1) +
per-tensor clip + Adam, the loop body of the reference Executor.train (wesep/utils/executor.py:70-134).
Prints ONE JSON line on rank 0.  `value`: inputs already resident in HBM; `e2e`: same step through
the public API from pinned host buffers (H2D every step, D2H of the loss every step).
--dump-outputs DIR: after the JSON line, rank 0 writes what the last timed (resident) step of each model block left to its
caller as DIR/<block>_{loss,grads}.npy (see `step_outputs`).  That step starts from the seeded initial state (`time_steps`),
so its inputs depend on the arguments only and two builds run with the same arguments can be compared array for array.
`roofline` describes the kernel with the LARGEST share of the timed step (shares from one CUPTI pass of a step inside this
run), `roofline.step` the whole step against the HBM roofline SURVEY.md 8d says binds it.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SPEX_ARGS = dict(B=256, H=512, L=20, N=256, P=3, R=4, X=8, spk_emb_dim=256, activate="relu", causal=False, norm="gLN",
                 skip_con=False, spk_fuse_type="concatConv", use_spk_transform=False, multi_fuse=True,
                 encoder_type="Multi", decoder_type="Multi", joint_training=True, multi_task=True, spksInTrain=251)
T_SAMPLES = 64000
METRIC = "utterances/sec Spex+ train step (4s@16kHz)"
BSRNN_ARGS = dict(sr=16000, win=512, stride=128, feature_dim=128, num_repeat=6, spk_fuse_type="multiply", use_spk_transform=False,
                  multi_fuse=False, joint_training=True, spk_model="ResNet34", spk_model_init=False,
                  spk_args=dict(feat_dim=80, embed_dim=256, pooling_func="TSTP", two_emb_layer=False), spk_emb_dim=256,
                  spk_model_freeze=False, spk_feat=True, feat_type="consistent", multi_task=False)   # bsrnn.yaml:46-83 verbatim
DPCCN_ARGS = dict(win=512, stride=128, feature_dim=257, tcn_blocks=10, tcn_layers=2, causal=False, spk_fuse_type="multiply",
                  use_spk_transform=False, multi_fuse=False, joint_training=True, spk_model="ResNet34", spk_model_init=False,
                  spk_args=dict(feat_dim=80, embed_dim=256, pooling_func="TSTP", two_emb_layer=False), spk_emb_dim=256,
                  spk_model_freeze=False, spk_feat=True, feat_type="consistent")                      # dpccn.yaml:40-80 verbatim
TFGRIDNET_ARGS = dict(n_srcs=1, sr=16000, n_fft=128, stride=64, window="hann", n_imics=1, n_layers=6, lstm_hidden_units=192,
                      attn_n_head=4, attn_approx_qk_dim=512, emb_dim=128, emb_ks=1, emb_hs=1, activation="prelu", eps=1.0e-5,
                      use_spk_transform=False, spk_fuse_type="multiply", joint_training=True, spk_model="ResNet34",
                      spk_model_init=False, spk_args=dict(feat_dim=80, embed_dim=256, pooling_func="TSTP", two_emb_layer=False),
                      spk_emb_dim=256, spk_model_freeze=False, spk_feat=True, feat_type="consistent")   # tfgridnet.yaml:42-84 minus multi_fuse
BSRNN_FBANK_FRAMES = 398        # 1 + (64000 - 400) // 160 frames of 25 ms / 10 ms fbank for a 4 s enrollment (SURVEY 8d config 3)
SPEX_BYTES_PER_ROW = 6.4e9      # algorithmic HBM bytes per row per train step (SURVEY.md 8d: 32 x 190 MB + 0.35 GB)
SPEX_FLOPS_PER_ROW = 396e9      # algorithmic flops per row per train step (132 GFLOP forward x 3)
BSRNN_FLOPS_PER_ROW = 1.02e12   # (340 GFLOP forward x 3)
DUMP_SAMPLE = 1 << 20           # --dump-outputs: at most this many elements per array (4 MiB fp32; 4 blocks = 16 MiB)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons),
                    samples=len(sm))


# ----------------------------------------------------------------------------- reference / CPU arm
def cpu_threads():
    """Intra-op threads for the CPU arm.  torch's CPU kernels on this model stop scaling (and then collapse:
    302 s/step with 128 threads vs 14 s/step with 8 on the same code) well below the box's core count, so the
    reference arm uses min(cores, 32) and says so in `cores`."""
    return max(1, min(os.cpu_count() or 1, 32))


def cpu_train_rows_per_s(rows, steps, warmup, threads):
    """The reference's algorithm on the host cores: oracle port (plain torch CPU fp32) of the same train
    step incl. reference-style per-tensor clip + Adam.  Bounded sample: `rows` model rows per step."""
    from oracle import losses as olosses
    from oracle import optim as ooptim
    from oracle import spexplus as ospex
    from wesep_b200 import synth
    torch.set_num_threads(threads)
    cfg = dict(ospex.DEFAULT_CFG)
    sd = ospex.make_state_dict(cfg)
    synth.fill_state_dict_(sd, seed=0)
    names = [k for k, v in sd.items() if v.is_floating_point() and "running_" not in k]
    P = [sd[k].requires_grad_(True) for k in names]
    m = [torch.zeros_like(p) for p in P]
    v = [torch.zeros_like(p) for p in P]
    b = synth.make_batch(rows, T=T_SAMPLES, Te=T_SAMPLES, seed=1234)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        bufs = {}
        out = ospex.convtasnet_forward(sd, cfg, b["wav_mix"], b["spk_embeds"], training=True, buffers_out=bufs)
        loss, _ = olosses.train_loss(out, b["wav_targets"], b["spk_label"])
        grads = [g.clone() for g in torch.autograd.grad(loss, P)]
        ooptim.clip_gradients(grads, 5.0)
        with torch.no_grad():
            ooptim.adam_step(P, grads, m, v, it + 1, 1e-3)
            sd.update(bufs)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    return rows / med, med, float(loss)


def cpu_model_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args, rank):
    """Reference arm: the reference's algorithm (oracle port of the Spex+ train step; the reference itself is a Python package
    that cannot be imported on the GPU box, DESIGN.md 8) on the host cores.  Every number printed is what actually ran."""
    if rank != 0:
        return
    threads = cpu_threads()
    rows = max(2, args.ref_rows)                    # >= 2 rows so the BatchNorm of the speaker encoder sees a batch
    steps, warm = args.steps, max(0, min(args.warmup, 1))
    val, med, loss = cpu_train_rows_per_s(rows, steps, warm, threads)
    sample = (f"{rows} rows x {T_SAMPLES} samples per step; ran {warm} warm-up + {steps} timed steps (median {med:.2f} s); "
              f"oracle port (plain torch fp32) on {threads} threads of {os.cpu_count()} host cores ({cpu_model_name()})")
    line = dict(metric=METRIC, value=val, unit="utterances/s", n_gpus=args.gpus, steps=steps, warmup=warm,
                steps_requested=args.steps, warmup_requested=args.warmup,
                ms_per_step=med * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload="Spex+ train step, 4s@16kHz, CPU sample of %d rows" % rows, rows_per_step=rows),
                cpu_baseline=dict(value=val, unit="utterances/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=val, unit="utterances/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0, loss=loss)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def kernel_shares(step_fn):
    """One CUPTI pass (torch.profiler) over one step: {kernel name: (count, total us)} and the total kernel time."""
    import collections
    from torch.profiler import ProfilerActivity, profile
    agg = collections.defaultdict(lambda: [0, 0.0])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step_fn()
        torch.cuda.synchronize()
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name
        if name.startswith("Memcpy") or name.startswith("Memset"):
            name = name.split(" ")[0]
        a = agg[name]
        a[0] += 1
        a[1] += ev.time_range.end - ev.time_range.start
    tot = sum(v[1] for v in agg.values())
    return agg, tot


# Per-launch algorithmic work of the Spex+ TCN-block kernels at n rows (B=256, H=512, K=6399; DESIGN.md 5) keyed by a
# substring of the kernel name: (bytes per row, flops per row, bound).  GEMMs execute 3x the algorithmic flops (3xTF32).
SPEX_KERNELS = {
    "gemm_dw_tc2_kernel<0, false>": (19.7e6, 1.677e9, "tensor"),      # dW1 += du . x^T
    "gemm_dw_tc2_kernel<1, true>": (19.7e6, 1.677e9, "tensor"),       # Gn = sum_t g . prelu(d)^T
    "gemm_wx_tc2_kernel<0, 10, 4>": (32.8e6, 1.677e9, "tensor"),      # B2
    "gemm_wx_tc2_kernel<2, 2, 4>": (26.2e6, 1.677e9, "tensor"),       # K4
    "gemm_wx_tc2_kernel<0, 2, 4>": (26.2e6, 1.677e9, "tensor"),       # B4
    "gemm_wx_tc2_kernel<0, 0, 6>": (19.7e6, 1.677e9, "tensor"),       # K2
    "tcn_dw_fwd": (26.2e6, 0.04e9, "hbm"),                            # K3
    "tcn_dw_bwd": (39.3e6, 0.1e9, "hbm"),                             # B3
}


def pick_roofline(agg, tot, table, rows, pk, passes, note):
    """The table kernel with the largest share of the step; achieved from its AVERAGE duration inside the step."""
    best = None
    for name, (cnt, us) in agg.items():
        for key, (byts, flops, bound) in table.items():
            if key in name and (best is None or us > best[2]):
                best = (name, key, us, cnt, byts, flops, bound)
    if best is None:
        return None
    name, key, us, cnt, byts, flops, bound = best
    sec = us / cnt * 1e-6
    if bound == "tensor":
        ach = passes * flops * rows / sec / 1e12
        peak, unit = pk["tf_sus"], "TFLOP/s"
    else:
        ach = byts * rows / sec / 1e9
        peak, unit = pk["hbm"], "GB/s"
    return dict(kernel=name[:90], share_of_step_kernel_time=us / tot, launches_per_step=cnt, avg_us=us / cnt, bound=bound,
                achieved=ach, peak=peak, unit=unit, frac=ach / peak, traffic=None,
                algorithmic_gbs=byts * rows / sec / 1e9, algorithmic_tflops=flops * rows / sec / 1e12, note=note)


def gpu_eager_baseline(n, dev):
    """The same-box incumbent (SURVEY.md 2.1): the reference's algorithm (oracle port = the reference's module graph) run by
    PyTorch eager on this B200 (cuDNN / cuBLAS, cudnn.benchmark as wesep/utils/utils.py:112), fp32 with TF32 off and on."""
    from oracle import losses as olosses
    from oracle import optim as ooptim
    from oracle import spexplus as ospex
    from wesep_b200 import synth
    out = {}
    torch.backends.cudnn.benchmark = True
    for tf32 in (False, True):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        rows = n
        while rows >= 2:
            try:
                cfg = dict(ospex.DEFAULT_CFG)
                sd = ospex.make_state_dict(cfg)
                synth.fill_state_dict_(sd, seed=0)
                sd = {k: v.to(dev) for k, v in sd.items()}
                names = [k for k, v in sd.items() if v.is_floating_point() and "running_" not in k]
                P = [sd[k].requires_grad_(True) for k in names]
                m = [torch.zeros_like(p) for p in P]
                v = [torch.zeros_like(p) for p in P]
                b = {k: x.to(dev) for k, x in synth.make_batch(rows, T=T_SAMPLES, Te=T_SAMPLES, seed=1234).items()}

                def step(it):
                    bufs = {}
                    o = ospex.convtasnet_forward(sd, cfg, b["wav_mix"], b["spk_embeds"], training=True, buffers_out=bufs)
                    loss, _ = olosses.train_loss(o, b["wav_targets"], b["spk_label"])
                    grads = list(torch.autograd.grad(loss, P))
                    ooptim.clip_gradients(grads, 5.0)
                    with torch.no_grad():
                        ooptim.adam_step(P, grads, m, v, it + 1, 1e-3)
                        sd.update(bufs)
                for it in range(2):
                    step(it)
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for it in range(3):
                    step(2 + it)
                e.record()
                torch.cuda.synchronize()
                ms = s.elapsed_time(e) / 3
                out["allow_tf32_%s" % str(tf32).lower()] = dict(value=rows / ms * 1e3, unit="utterances/s", rows=rows, ms_per_step=ms)
                break
            except torch.OutOfMemoryError:
                rows //= 2
            finally:
                P = m = v = sd = b = None
                torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = True
    out["what"] = ("oracle port (the reference's op graph in plain torch) run eagerly on this GPU: 2 warm-up + 3 timed steps, "
                   "cudnn.benchmark=True; the reference's own GPU path uses PyTorch defaults (cudnn TF32 on, matmul TF32 off)")
    return out


def time_steps(one, warmup, steps, barrier, world, dev, restore=None):
    """`warmup` untimed steps, then `steps` timed ones.  `restore()` runs between the two timed windows, right before the last
    step: it puts the model back into the seeded state it started from, so what that step computes depends on the arguments
    only.  (The kernels accumulate in fp32 with atomics, so every step is reproducible to rounding; Adam's first updates move
    each element by about +-lr according to its gradient's sign, which would turn that rounding into differences of order lr
    after a few steps.)"""
    from wesep_b200 import _lib
    import torch.distributed as dist
    for _ in range(warmup):
        one()
    barrier()
    l0 = _lib.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ev[0].record()
    for _ in range(steps - 1):
        one()
    ev[1].record()
    if restore is not None:
        restore()
    ev[2].record()
    last = one()
    ev[3].record()
    barrier()
    ms = ev[0].elapsed_time(ev[1]) + ev[2].elapsed_time(ev[3])
    launches = _lib.launch_count() - l0
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt)
    return ms, launches, float(last)


def _dump_sample(x):
    """x (flat, on the device) as an fp32 host array; beyond DUMP_SAMPLE elements, the same seeded sample of indices for a
    given length."""
    if x.numel() > DUMP_SAMPLE:
        import numpy as np
        idx = np.sort(np.random.default_rng(0).choice(x.numel(), DUMP_SAMPLE, replace=False))
        x = x[torch.from_numpy(idx).to(x.device)]
    return x.float().cpu().numpy()


def step_outputs(opt, loss):
    """What a train step computes for its caller: the loss and the gradients the optimizer applied (in parameter order).  The
    updated parameters are left out: Adam's step from the seeded state moves every element by about +-lr by the sign of its
    gradient, and for elements whose gradient is at rounding level (e.g. the exactly-zero decoder-bias gradients of the
    shift-invariant SI-SDR) that sign is itself rounding."""
    import numpy as np
    with torch.no_grad():
        grads = torch.cat([p.grad.reshape(-1) for p in opt.arena.params])
    return dict(loss=np.array([loss], np.float64), grads=_dump_sample(grads))


def write_outputs(out_dir, blocks):
    """blocks: {block name: step_outputs(...)} -> out_dir/<block>_<array>.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for block, arrays in blocks.items():
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, f"{block}_{name}.npy"), a)


def run_pbsrnn(args, rank, world, dev, pk, barrier, dumps):
    """BASELINE config 3: pBSRNN train step, 4 s @ 16 kHz, 16 rows per GPU, bsrnn.yaml network (speaker embeddings as input)."""
    import numpy as np
    from wesep_b200 import _lib, ops, synth
    from wesep_b200.distributed import GradAllReducer, broadcast_params
    from wesep_b200.models import get_model
    from wesep_b200.utils.executor import restore_train_state, snapshot_train_state
    from wesep_b200.utils.optim import FusedClipAdam
    n = args.bsrnn_rows
    torch.manual_seed(42 + rank)
    model = get_model("BSRNN")(**BSRNN_ARGS).to(dev).train()
    opt = FusedClipAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, clip=5.0)
    broadcast_params(opt.arena.flat_p)
    reducer = GradAllReducer(opt.arena.flat_g, n_buckets=1) if world > 1 else None
    host = synth.make_batch(n, T=T_SAMPLES, Te=8, seed=4321 + rank, pin=True)
    emb_h = torch.from_numpy(np.random.default_rng(5 + rank).standard_normal((n, BSRNN_FBANK_FRAMES, 80))
                             .astype(np.float32)).pin_memory()          # enrollment fbank features (after CMN) ~ N(0, 1)
    host = dict(wav_mix=host["wav_mix"], wav_targets=host["wav_targets"], emb=emb_h)
    resident = {k: v.to(dev) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def step(batch, read_loss):
        mix = batch["wav_mix"].to(dev, non_blocking=True)
        tgt = batch["wav_targets"].to(dev, non_blocking=True)
        emb = batch["emb"].to(dev, non_blocking=True)
        opt.zero_grad()
        est, _ = model(mix, emb)
        losses, _ = ops.sisdr_losses([est], tgt)
        losses[0].backward()
        if reducer is not None:
            reducer.all_reduce()
            opt.grad_scale = reducer.grad_scale
        opt.step()
        return losses[0].item() if read_loss else losses[0]

    graphed = None
    if world == 1 and not args.no_graph:
        # the eager pBSRNN step is host-bound (~4000 launches incl. the per-band loops): capture it once, replay per step
        from wesep_b200.utils.executor import GraphedStep

        def body(b):
            est, _ = model(b["wav_mix"], b["emb"])
            losses, _ = ops.sisdr_losses([est], b["wav_targets"])
            losses[0].backward()
            return losses[0]
        graphed = GraphedStep(model, opt, resident, body, warmup=2)

        def step(batch, read_loss):                                # noqa: F811
            loss = graphed(batch)                                   # copies the batch (pinned host or device) into the static inputs
            return loss.item() if read_loss else loss

    seed = snapshot_train_state(model, opt)

    def restore():
        restore_train_state(model, opt, seed)
    ms_res, launches, loss_res = time_steps(lambda: step(resident, False), args.warmup, args.steps, barrier, world, dev, restore)
    if args.dump_outputs and rank == 0:
        dumps["pbsrnn"] = step_outputs(opt, loss_res)
    if graphed is not None:
        launches = graphed.launches_per_step * args.steps
    ms_e2e, _, loss_e2e = time_steps(lambda: step(host, True), 1, args.steps, barrier, world, dev, restore)
    if rank != 0:
        step(resident, False)          # the CUPTI pass below is one more COLLECTIVE step: every rank takes part
        barrier()
        return None
    agg, tot = kernel_shares(lambda: step(resident, False))
    barrier()
    rec = {k: v for k, v in agg.items() if "lstm_rec" in k}
    rec_us = sum(v[1] for v in rec.values())
    rec_n = sum(v[0] for v in rec.values())
    # one launch of either recurrence kernel: 2 directions x (4 Hd x Hd) x (sequences x steps) MACs; Q S is the same for
    # band_rnn (32 n x 501) and band_comm (501 n x 32)
    Hd, QS = 256, 32 * n * 501
    alg = 2.0 * 2 * 4 * Hd * Hd * QS
    sec = rec_us / max(rec_n, 1) * 1e-6
    top = sorted(agg.items(), key=lambda kv: -kv[1][1])[:6]
    step_tf = 3 * BSRNN_FLOPS_PER_ROW * n * args.steps / (ms_res * 1e-3) / 1e12
    roof = dict(kernel="lstm_rec_fwd_kernel / lstm_rec_bwd_kernel (persistent cluster BLSTM recurrence, tcgen05 kind::f16)",
                share_of_step_kernel_time=rec_us / tot, launches_per_step=rec_n, avg_us=rec_us / max(rec_n, 1), bound="tensor",
                achieved=3 * alg / sec / 1e12, peak=pk["tf_sus"], unit="TFLOP/s", frac=3 * alg / sec / 1e12 / pk["tf_sus"],
                traffic=None, algorithmic_tflops=alg / sec / 1e12,
                serial_floor_us_per_step=1.65,
                note="executed = 3 x algorithmic flops (fp16 / bf16 hi+lo split products, fp32-grade); avg over the 24 launches of a "
                     "step (6 layers x (band_rnn 501 steps + band_comm 32 steps) x (fwd + bwd)); peak = measured sustained bf16 (%s); "
                     "serial floor per time step of one cluster = one group's step product on the tensor pipe (48 MMAs x 32 clk) + "
                     "one DSMEM all-gather hop + the cell's dependent MUFU chain ~ 3100 clk (DESIGN.md)" % pk["src"],
                step=dict(bound="tensor", achieved=step_tf, peak=pk["tf_sus"], unit="TFLOP/s", frac=step_tf / pk["tf_sus"],
                          note="whole step, per GPU: 3 x 1.02 TFLOP per row (SURVEY 8d, fp32-grade split products) x rows / step time "
                               "/ sustained bf16 peak"))
    return dict(metric="utterances/sec pBSRNN train step (4s@16kHz)", value=n * world * args.steps / (ms_res * 1e-3),
                unit="utterances/s", ms_per_step=ms_res / args.steps, rows_per_gpu=n, global_rows=n * world,
                config=dict(workload="pBSRNN (BSRNN, examples/librimix/tse/v2/confs/bsrnn.yaml network: 32 bands, feature 128, "
                                     "hidden 256, 6 BSNet repeats, multiply fusion, jointly trained wespeaker ResNet34-TSTP speaker encoder on "
                                     "[n, 398, 80] enrollment fbank features) full train step, 4s@16kHz, %d rows per GPU" % n,
                            loss="SI-SDR", optimizer="per-tensor clip 5.0 + Adam(wd 1e-4)",
                            launch="one CUDA-graph replay per step" if graphed is not None else "eager (one launch per kernel)",
                            gemm_mode="GEMMs: mixed split (tf32 hi*hi + 2 bf16 cross terms) / 3xTF32; recurrence fp16 hi/lo (fwd) / bf16 hi/lo "
                                      "(bwd) split products"),
                e2e=dict(value=n * world * args.steps / (ms_e2e * 1e-3), unit="utterances/s", h2d_bytes_per_step=h2d,
                         d2h_bytes_per_step=4, ms_per_step=ms_e2e / args.steps),
                gpu_launches=launches, loss=loss_res, loss_e2e=loss_e2e, roofline=roof,
                top_kernels=[dict(kernel=k[:70], share=v[1] / tot, count=v[0]) for k, v in top])


def run_extra(args, dev, which, dumps):
    """Further blocks (single GPU only): pDPCCN (SURVEY.md 8 row a23) and TF-GridNet (row a24, BASELINE config 5) train steps on
    the recipe networks verbatim (jointly trained ResNet34 on fbank features), 4 s @ 16 kHz, eager launches."""
    import numpy as np
    from wesep_b200 import _lib, ops, synth
    from wesep_b200.models import get_model
    from wesep_b200.utils.executor import restore_train_state, snapshot_train_state
    from wesep_b200.utils.optim import FusedClipAdam
    n = args.dpccn_rows if which == "DPCCN" else args.tfgridnet_rows
    torch.manual_seed(42)
    model = get_model(which)(**(DPCCN_ARGS if which == "DPCCN" else TFGRIDNET_ARGS)).to(dev).train()
    opt = FusedClipAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, clip=5.0)
    host = synth.make_batch(n, T=T_SAMPLES, Te=8, seed=777, pin=True)
    emb_h = torch.from_numpy(np.random.default_rng(6).standard_normal((n, BSRNN_FBANK_FRAMES, 80)).astype(np.float32)).pin_memory()
    host = dict(wav_mix=host["wav_mix"], wav_targets=host["wav_targets"], emb=emb_h)
    resident = {k: v.to(dev) for k, v in host.items()}

    def step(batch, read_loss):
        mix = batch["wav_mix"].to(dev, non_blocking=True)
        tgt = batch["wav_targets"].to(dev, non_blocking=True)
        emb = batch["emb"].to(dev, non_blocking=True)
        opt.zero_grad()
        est, _ = model(mix, emb)
        losses, _ = ops.sisdr_losses([est], tgt)
        losses[0].backward()
        opt.step()
        return losses[0].item() if read_loss else losses[0]

    K = args.steps

    def sync():
        torch.cuda.synchronize(dev)

    graphed = None
    if not args.no_graph:
        try:                                                      # the eager step is host-bound (thousands of small launches)
            from wesep_b200.utils.executor import GraphedStep

            def body(b):
                est, _ = model(b["wav_mix"], b["emb"])
                losses, _ = ops.sisdr_losses([est], b["wav_targets"])
                losses[0].backward()
                return losses[0]
            graphed = GraphedStep(model, opt, resident, body, warmup=2)
            eager_step = step

            def step(batch, read_loss):                            # noqa: F811
                loss = graphed(batch)
                return loss.item() if read_loss else loss
        except Exception as ex:                                    # capture is an optimisation: fall back to eager launches
            graphed, graph_error = None, repr(ex)[:200]
            torch.cuda.synchronize(dev)
    seed = snapshot_train_state(model, opt)

    def restore():
        restore_train_state(model, opt, seed)
    ms_res, launches, loss_res = time_steps(lambda: step(resident, False), 3, K, sync, 1, dev, restore)
    if args.dump_outputs:
        dumps[which.lower()] = step_outputs(opt, loss_res)
    ms_e2e, _, loss_e2e = time_steps(lambda: step(host, True), 1, K, sync, 1, dev, restore)
    if graphed is not None:
        launches = graphed.launches_per_step * K
    agg, tot = kernel_shares(lambda: step(resident, False))
    top = sorted(agg.items(), key=lambda kv: -kv[1][1])[:6]
    if which == "DPCCN":
        metric = "utterances/sec pDPCCN train step (4s@16kHz)"
        cfg = dict(workload="pDPCCN (examples/librimix/tse/v2/confs/dpccn.yaml network: 257 bins, dense conv encoder / "
                            "decoder, 2 x 10 TCN blocks, multiply fusion, jointly trained wespeaker ResNet34-TSTP on [n, 398, 80] "
                            "fbank features) full train step, 4s@16kHz, %d rows" % n,
                   conv="3x3 (transposed) convolutions = im2col / col2im + tcgen05 pointwise GEMM")
    else:
        metric = "utterances/sec TF-GridNet train step (4s@16kHz)"
        cfg = dict(workload="TF-GridNet (examples/librimix/tse/v2/confs/tfgridnet.yaml network: n_fft 128, 6 GridNet blocks, 128 "
                            "channels, BLSTM hidden 192, 4 heads, multiply fusion, jointly trained wespeaker ResNet34-TSTP on "
                            "[n, 398, 80] fbank features) full train step, 4s@16kHz, %d rows (BASELINE config 5)" % n,
                   blstm="persistent cluster recurrence kernel (hidden 192, 6 CTAs per cluster)",
                   attention="two pointwise GEMMs + row softmax per (batch, head)")
    out = dict(metric=metric, value=n * K / (ms_res * 1e-3), unit="utterances/s",
               ms_per_step=ms_res / K, steps=K, rows_per_gpu=n,
               config=dict(cfg, loss="SI-SDR", optimizer="per-tensor clip 5.0 + Adam(wd 1e-4)",
                           launch="one CUDA-graph replay per step" if graphed is not None else "eager (one launch per kernel)"),
               e2e=dict(value=n * K / (ms_e2e * 1e-3), unit="utterances/s",
                        h2d_bytes_per_step=sum(v.numel() * v.element_size() for v in host.values()), d2h_bytes_per_step=4,
                        ms_per_step=ms_e2e / K),
               gpu_launches=launches, loss=loss_res, loss_e2e=loss_e2e, peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 2 ** 30,
               top_kernels=[dict(kernel=k[:70], share=v[1] / tot, count=v[0]) for k, v in top])
    del model, opt, resident, seed
    torch.cuda.empty_cache()
    return out


def run_ours(args, rank, world, local):
    from wesep_b200 import _lib, synth
    from wesep_b200.distributed import GradAllReducer, broadcast_params
    from wesep_b200.models import get_model
    from wesep_b200.utils.executor import restore_train_state, snapshot_train_state, train_step
    from wesep_b200.utils.lr import exponential_decrease_lr, set_lr
    from wesep_b200.utils.optim import FusedClipAdam
    import torch.distributed as dist

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pk = peaks()
    n = args.rows
    torch.manual_seed(42 + rank)                                # train.py:88 per-rank seed
    model = get_model("ConvTasNet")(**SPEX_ARGS).to(dev).train()
    opt = FusedClipAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, clip=5.0)
    broadcast_params(opt.arena.flat_p)
    reducer = GradAllReducer(opt.arena.flat_g, n_buckets=3) if world > 1 else None
    host = synth.make_batch(n, T=T_SAMPLES, Te=T_SAMPLES, seed=1234 + rank, pin=True)
    resident = {k: v.to(dev) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    graphed = None
    if args.cuda_graph:
        if world > 1:
            raise SystemExit("--cuda-graph is single-process (the gradient all-reduce is not captured)")
        from wesep_b200.utils.executor import GraphedTrainStep
        graphed = GraphedTrainStep(model, opt, resident, warmup=3)   # 3 eager steps, then ONE capture of the whole step

    it = [0]

    def one(batch, read_loss):
        set_lr(opt, exponential_decrease_lr(it[0], 150 * 1000, 1e-3, 2.5e-5))
        it[0] += 1
        loss = graphed(batch) if graphed is not None else train_step(model, batch, opt, reducer)
        return loss.item() if read_loss else loss               # .item() = D2H of the step's result

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    seed = snapshot_train_state(model, opt)

    def restore():
        restore_train_state(model, opt, seed)
    ms_res, launches, loss_res = time_steps(lambda: one(resident, False), args.warmup, args.steps, barrier, world, dev, restore)
    dumps = {}
    if args.dump_outputs and rank == 0:
        dumps["spex"] = step_outputs(opt, loss_res)
    if graphed is not None:                                     # replays do not pass through the host-side counter
        launches = graphed.launches_per_step * args.steps
    ms_e2e, _, loss_e2e = time_steps(lambda: one(host, True), args.warmup, args.steps, barrier, world, dev, restore)
    clocks_spex = sampler.summary() if sampler else None
    value = n * world * args.steps / (ms_res * 1e-3)
    e2e = n * world * args.steps / (ms_e2e * 1e-3)
    roof = None
    if rank != 0:
        one(resident, False)           # the CUPTI pass of rank 0 is one more COLLECTIVE step: every rank takes part
    if rank == 0:
        agg, tot = kernel_shares(lambda: one(resident, False))
        roof = pick_roofline(agg, tot, SPEX_KERNELS, n, pk, 3,
                             "kernel with the largest share of one timed step (CUPTI pass inside this run); achieved = executed "
                             "tensor flops (3 x algorithmic: fp32-grade split products) / its average duration INSIDE the step / "
                             "measured sustained bf16 peak (%s); kernels without a per-channel prologue (<0, *, *>) run the mixed "
                             "split = one kind::tf32 product (half the bf16 rate) + two bf16 cross terms = 3 products in 4 "
                             "bf16-time units, ceiling 0.75; the <2|3, *, *> kernels run 3xTF32, ceiling 0.5; traffic: see "
                             "profiles/ (ncu dram bytes ~ algorithmic bytes)" % pk["src"])
        if roof is not None:
            step_gbs = SPEX_BYTES_PER_ROW * n * args.steps / (ms_res * 1e-3) / 1e9
            roof["step"] = dict(bound="hbm", achieved=step_gbs, peak=pk["hbm"], unit="GB/s", frac=step_gbs / pk["hbm"],
                                note="whole train step: 6.4 GB algorithmic bytes per row (SURVEY 8d) x rows / step time / measured HBM "
                                     "copy bandwidth - the binding roofline of the Spex+ step")
            roof["top_kernels"] = [dict(kernel=k[:70], share=v[1] / tot, count=v[0])
                                   for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])[:6]]
    barrier()
    # free the Spex+ state before the second model
    del model, opt, reducer, resident, graphed, seed
    torch.cuda.empty_cache()
    pb = None
    if not args.no_pbsrnn:
        pb = run_pbsrnn(args, rank, world, dev, pk, barrier, dumps)
    if rank != 0:
        return
    dp = None
    if world == 1 and not args.no_dpccn:
        try:
            dp = run_extra(args, dev, "DPCCN", dumps)
        except Exception as ex:                                 # extra block: never lose the bench line over it
            dp = dict(error=repr(ex)[:300])
    tg = None
    if world == 1 and not args.no_tfgridnet:
        try:
            tg = run_extra(args, dev, "TFGridNet", dumps)
        except Exception as ex:
            tg = dict(error=repr(ex)[:300])
    cpu = eager = None
    if world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        rows = max(2, args.ref_rows)
        v, med, _ = cpu_train_rows_per_s(rows, 2, 1, threads)
        cpu = dict(value=v, unit="utterances/s", cores=threads, kind="port",
                   sample=f"{rows} rows x {T_SAMPLES} samples, 1 warm-up + 2 timed steps (median {med:.2f} s), "
                          f"oracle port (plain torch fp32) on {threads} threads of {os.cpu_count()} host cores ({cpu_model_name()})")
        try:
            eager = gpu_eager_baseline(n, dev)
        except Exception as ex:                                 # informative block: never lose the bench line over it
            eager = dict(error=repr(ex)[:200])
    line = dict(
        metric=METRIC, value=value, unit="utterances/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_res / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
        data="synthetic", impl="ours",
        config=dict(workload="Spex+ (ConvTasNet, examples/librimix/tse/v2/confs/spexplus.yaml) full train step, "
                             "4s@16kHz, %d model rows per GPU" % n,
                    rows_per_gpu=n, global_rows=n * world, samples=T_SAMPLES, parallelism="dp%d" % world,
                    gemm_mode="fp32-grade split products on tcgen05 (cta_group::2, TMA, TMEM): tf32 hi*hi + 2 bf16 cross terms (mixed), "
                              "3xTF32 where a per-channel prologue rewrites the operand; mma.sync for odd shapes",
                    l2="inputs and activations >> L2 (126 MB)",
                    loss="0.8/0.1/0.1 SI-SDR + 0.5 CE", optimizer="per-tensor clip 5.0 + Adam(wd 1e-4), exp-decay lr",
                    launch="one CUDA-graph replay per step" if args.cuda_graph else "eager (one launch per kernel)"),
        e2e=dict(value=e2e, unit="utterances/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
                 ms_per_step=ms_e2e / args.steps),
        gpu_launches=launches, clocks=clocks_spex, loss=loss_res, loss_e2e=loss_e2e,
        roofline=roof, pbsrnn=pb, dpccn=dp, tfgridnet=tg, cpu_baseline=cpu, gpu_eager_baseline=eager)
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, dumps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every model block (and of the --impl reference arm)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=32, help="Spex+ model rows (utterances) per GPU per step")
    ap.add_argument("--bsrnn-rows", type=int, default=16, help="pBSRNN model rows per GPU per step")
    ap.add_argument("--ref-rows", type=int, default=2, help="rows per step of the bounded CPU sample (>= 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU and GPU-eager baselines")
    ap.add_argument("--no-pbsrnn", action="store_true", help="skip the pBSRNN block")
    ap.add_argument("--no-dpccn", action="store_true", help="skip the pDPCCN block (single-GPU runs only)")
    ap.add_argument("--dpccn-rows", type=int, default=4, help="pDPCCN block: model rows")
    ap.add_argument("--no-tfgridnet", action="store_true", help="skip the TF-GridNet block (single-GPU runs only)")
    ap.add_argument("--tfgridnet-rows", type=int, default=4, help="TF-GridNet block: model rows (BASELINE config 5: 4)")
    ap.add_argument("--no-graph", action="store_true", help="pBSRNN block: eager launches instead of a CUDA-graph replay per step")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="capture the whole Spex+ train step in a CUDA graph and time replays (single GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of each block's last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a GPU (no CPU fallback)")
    from wesep_b200.distributed import init_from_env
    rank, world, local = init_from_env("nccl")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    run_ours(args, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
