"""Train-step driver — mirrors the loop body of the reference Executor.train
(wesep/utils/executor.py:70-134): forward, weighted SI-SDR (+CE) loss, backward, gradient
all-reduce, per-tensor clip + Adam.  Host syncs per step: only the caller's optional loss read."""
import torch

from wesep_b200 import ops


_LOSS_W = {}


def compute_loss(outputs, targets, spk_label, loss_posi=((0, 1, 2), (3,)), loss_weight=((0.8, 0.1, 0.1), (0.5,)),
                 multi_task=True):
    """loss = sum_j w0[j] * SISDR(outputs[posi0[j]], targets) (+ w1[j] * CE(outputs[posi1[j]], spk_label))
    — executor.py:105-122 with criterion = [SISDR, CE]; all SI-SDR terms in one fused kernel."""
    if not isinstance(outputs, (list, tuple)):
        outputs = [outputs]
    ests = [outputs[p] for p in loss_posi[0]]
    L = ests[0].shape[-1]
    tgt = targets if targets.shape[-1] == L else targets[:, :L]
    losses, rows = ops.sisdr_losses(ests, tgt)
    key = (tuple(float(v) for v in loss_weight[0]), losses.device)
    w = _LOSS_W.get(key)
    if w is None:       # cached: a pageable host->device copy per step would also forbid CUDA-graph capture
        w = _LOSS_W[key] = torch.tensor(list(key[0]), dtype=torch.float32, device=losses.device)
    loss = (losses * w).sum()
    if multi_task and len(loss_posi) > 1:
        for j, p in enumerate(loss_posi[1]):
            loss = loss + loss_weight[1][j] * ops.cross_entropy(outputs[p], spk_label)
    return loss, rows


def train_step(model, batch, optimizer, reducer=None, loss_posi=((0, 1, 2), (3,)), loss_weight=((0.8, 0.1, 0.1), (0.5,)),
               multi_task=True, device=None):
    """One iteration of Executor.train. `batch` holds wav_mix / wav_targets / spk_embeds / spk_label
    (host pinned or device tensors). Returns the (device) loss tensor; no host sync here."""
    if device is None:
        device = next(model.parameters()).device
    features = batch["wav_mix"].to(device, non_blocking=True).float()
    targets = batch["wav_targets"].to(device, non_blocking=True).float()
    enroll = batch["spk_embeds"].to(device, non_blocking=True).float()
    spk_label = batch["spk_label"].to(device, non_blocking=True)
    optimizer.zero_grad()
    outputs = model(features, enroll)
    loss, _ = compute_loss(outputs, targets, spk_label, loss_posi, loss_weight, multi_task)
    with ops.direct_param_grads():  # TCN-block kernels accumulate straight into the optimizer's gradient arena
        loss.backward()
    if reducer is not None:
        reducer.all_reduce()
        optimizer.grad_scale = reducer.grad_scale
    optimizer.step()
    return loss


def snapshot_train_state(model, optimizer):
    """Copies of everything a train step updates: parameters, Adam moments and step counter, module buffers."""
    return dict(p=optimizer.arena.flat_p.clone(), m=optimizer.exp_avg.clone(), v=optimizer.exp_avg_sq.clone(),
                step=optimizer.step_count, bufs={k: b.clone() for k, b in model.named_buffers()})


def restore_train_state(model, optimizer, snap):
    """Puts a snapshot_train_state() back in place (same storage, so CUDA graphs keep seeing it)."""
    with torch.no_grad():
        optimizer.arena.flat_p.copy_(snap["p"])
        optimizer.exp_avg.copy_(snap["m"])
        optimizer.exp_avg_sq.copy_(snap["v"])
        optimizer.step_count = snap["step"]
        for k, b in model.named_buffers():
            b.copy_(snap["bufs"][k])


class GraphedStep:
    """A whole train step (zero_grad, forward, loss, backward, clip + Adam) captured ONCE in a CUDA graph and replayed:
    the ~10^3 kernel launches of a step become one graph launch, removing the inter-kernel gaps and all per-step Python /
    ctypes work (the pBSRNN step is otherwise host-bound).  Single-process only (the gradient all-reduce stays outside a
    graph: use the eager step with a reducer for N > 1).  Shapes are frozen at capture: every batch must match the example.

        step = GraphedStep(model, optimizer, example_batch, body)    # body(static_batch) -> loss, up to and incl. backward
        loss = step(batch)                                            # device tensor (static storage): read or copy it

    The constructor runs `warmup` eager steps (every lazily created buffer must exist before the capture) and then RESTORES
    parameters, Adam moments, the step counter and all module buffers, so training starts from the state it was given.
    The learning rate may change between calls (`param_groups[0]["lr"]`): the optimizer kernels read the schedule-dependent
    scalars from device memory (`FusedClipAdam.enable_device_scalars`)."""

    def __init__(self, model, optimizer, example_batch, body, warmup=3):
        self.model, self.opt, self.body = model, optimizer, body
        dev = next(model.parameters()).device
        self.static = {k: v.to(dev).clone() for k, v in example_batch.items()}
        optimizer.enable_device_scalars()
        snap = snapshot_train_state(model, optimizer)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                      # warm-up off the default stream, as graph capture requires
            for _ in range(warmup):
                optimizer.push_scalars()
                self._body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        restore_train_state(model, optimizer, snap)
        self.graph = torch.cuda.CUDAGraph()
        l0 = ops._lib.launch_count()
        with torch.cuda.graph(self.graph):
            self.loss = self._body()
        self.launches_per_step = ops._lib.launch_count() - l0   # kernels of this library inside one replay
        restore_train_state(model, optimizer, snap)        # (capture does not execute, but keep the invariant explicit)

    def _body(self):
        self.opt.zero_grad()
        loss = self.body(self.static)
        self.opt.launch()
        return loss

    def __call__(self, batch):
        for k, v in self.static.items():
            v.copy_(batch[k], non_blocking=True)            # pinned host or device source (dtype cast by copy_)
        self.opt.push_scalars()
        self.graph.replay()
        return self.loss


class GraphedTrainStep(GraphedStep):
    """GraphedStep for the Spex+ recipe loop body (weighted SI-SDR + CE loss on the four-tensor collate batch)."""

    def __init__(self, model, optimizer, example_batch, loss_posi=((0, 1, 2), (3,)), loss_weight=((0.8, 0.1, 0.1), (0.5,)),
                 multi_task=True, warmup=3):
        # only the four tensors the step consumes (a reference collate batch also carries `spk` / `key` lists), cast as
        # train_step casts them
        ex = {k: example_batch[k].float() for k in ("wav_mix", "wav_targets", "spk_embeds")}
        ex["spk_label"] = example_batch["spk_label"]

        def body(b):
            outputs = model(b["wav_mix"], b["spk_embeds"])
            loss, _ = compute_loss(outputs, b["wav_targets"], b["spk_label"], loss_posi, loss_weight, multi_task)
            with ops.direct_param_grads():
                loss.backward()
            return loss
        super().__init__(model, optimizer, ex, body, warmup)


class Executor:
    """reference wesep/utils/executor.py:27-152 (train only; logging left to the caller)."""

    def __init__(self):
        self.step = 0

    def train(self, dataloader, models, epoch_iter, optimizers, criterion, schedulers, scaler, epoch, enable_amp,
              logger, clip_grad=5.0, log_batch_interval=100, device=torch.device("cuda"), se_loss_weight=1.0,
              multi_task=False, reducer=None, SSA_enroll_prob=0, fbank_args=None, sample_rate=16000, speaker_feat=True):
        if enable_amp:
            raise NotImplementedError("AMP is off in every recipe (fp32 path only)")
        if SSA_enroll_prob and SSA_enroll_prob > 0:
            raise NotImplementedError("SSA_enroll_prob > 0 (self-enrollment second pass, executor.py:92-104) is not built")
        names = [type(c).__name__ for c in (criterion or [])]
        if criterion is not None and not (names[:1] == ["SISDRLoss"] and all(n == "CrossEntropyLoss" for n in names[1:])):
            raise NotImplementedError(f"criterion {names}: the fused loss covers SISDR (+ CE) only")
        model, optimizer, scheduler = models[0], optimizers[0], schedulers[0]
        model.train()
        optimizer.param_groups[0]["clip"] = clip_grad or 0.0
        losses = []
        for i, batch in enumerate(dataloader):
            cur_iter = (epoch - 1) * epoch_iter + i
            scheduler.step(cur_iter)
            loss = train_step(model, batch, optimizer, reducer, se_loss_weight[0], se_loss_weight[1], multi_task, device)
            losses.append(loss.item())
            if logger is not None and (i + 1) % log_batch_interval == 0:
                logger.info("TRAIN epoch %d iter %d loss %.4f lr %.3e" % (epoch, i + 1, sum(losses) / len(losses),
                                                                           optimizer.param_groups[0]["lr"]))
            if (i + 1) == epoch_iter:
                break
        return sum(losses) / len(losses), 0
