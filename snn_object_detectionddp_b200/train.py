"""Epoch loops of the reference (train.py:46-241) on the B200 path: same function names, same TensorBoard tags, same
checkpoint files -- without the reference's 3-5 host synchronisations per batch.

    reference                                      here
    ---------------------------------------------  ----------------------------------------------------------------
    per batch: scalar_loss.item() x2, 3x            loss items stay on the device; `DeviceMetrics` keeps the running totals
      loss_components[i].item(), pbar, writer         and a ring of the last N steps' (items, lr) on the device and reads
      (train.py:81-100)                                them back ONCE every N steps, then emits the same per-batch scalars
                                                       with the same global_step values
    optimizer / scheduler built in train_loop       `Trainer` (fused clip + AdamW over the flat buffers, tabulated OneCycle)
      (train.py:155-169)
    DataLoader(shuffle=True) (main.py:57-72)        `ShardedSampler`: per-rank shard of the sequence-grouped split

TensorBoard tags (train.py:88-100, 137-143, 211-226), unchanged:
    Loss/train_batch, Train_Loss_Components_Batch/{box,cls,dfl}_loss_batch, LearningRate/batch,
    Loss/val_batch, Val_Loss_Components_Batch/{box,cls,dfl}_loss_batch,
    Loss/train, Loss/val, LearningRate, Train_Loss_Components/{box,cls,dfl}_loss, Val_Loss_Components/{box,cls,dfl}_loss
"""
import math
import os
from collections import defaultdict

import torch

from .data import custom_collate_fn  # noqa: F401  (main.py:10 imports it from `train`)

COMPONENTS = ("box_loss", "cls_loss", "dfl_loss")


class DeviceMetrics:
    """Loss bookkeeping of train_one_epoch / validate_one_epoch (train.py:52-53, 81-83, 102-104) without per-batch syncs.

    `update(items, step, lr, scale)` enqueues a few tiny device ops (no host read); `flush()` copies the ring of pending
    steps to the host once and returns [(global_step, items[3], lr, scalar)]; `averages(n_batches)` is the epoch return
    value of the reference: (total_loss / n, total_components / n).  `scale`: the reference's TRAINING scalar is
    `loss_components.sum()` with loss_components = loss * batch_size (train.py:74-75), its VALIDATION scalar is
    `loss_components_detached.sum()` (train.py:127) -- scale = B resp. 1."""

    def __init__(self, device, every=50):
        self.device, self.every = torch.device(device), max(1, int(every))
        self.total = torch.zeros(4, device=self.device, dtype=torch.float64)       # components[3], scalar
        self.ring = torch.zeros(self.every, 5, device=self.device, dtype=torch.float32)
        self.steps, self.n = [], 0

    def update(self, items, global_step, lr=0.0, scale=1.0):
        slot = len(self.steps)
        it = items.detach()
        self.ring[slot, :3].copy_(it, non_blocking=True)
        self.ring[slot, 3] = lr
        self.ring[slot, 4] = it.sum() * scale
        self.total[:3] += it.double()
        self.total[3] += self.ring[slot, 4].double()
        self.steps.append(int(global_step))
        self.n += 1
        return len(self.steps) >= self.every

    def flush(self):
        if not self.steps:
            return []
        host = self.ring[:len(self.steps)].cpu()          # the ONE synchronisation per `every` steps
        out = [(g, host[i, :3].clone(), float(host[i, 3]), float(host[i, 4])) for i, g in enumerate(self.steps)]
        self.steps = []
        return out

    def averages(self, n_batches):
        tot = (self.total / max(1, n_batches)).float().cpu()
        return float(tot[3]), tot[:3]


def _log_batches(writer, rows, train):
    if writer is None:
        return
    tag_loss, tag_comp = ("Loss/train_batch", "Train_Loss_Components_Batch") if train else ("Loss/val_batch", "Val_Loss_Components_Batch")
    for gstep, items, lr, scalar in rows:
        writer.add_scalar(tag_loss, scalar, gstep)
        writer.add_scalars(tag_comp, {"box_loss_batch": float(items[0]), "cls_loss_batch": float(items[1]),
                                      "dfl_loss_batch": float(items[2])}, gstep)
        if train:
            writer.add_scalar("LearningRate/batch", lr, gstep)


def _batch_dict(trainer, labels_tensor, batch_size, max_boxes):
    return trainer.prepare_batch(labels_tensor, batch_size, max_boxes=max_boxes)


def train_one_epoch(trainer, dataloader, sequence_length=None, writer=None, epoch=0, log_every=50, max_boxes=None, graphed=False,
                    prefetcher=None):
    """reference train.py:46-104.  `trainer` = trainer.Trainer (it owns model, loss, optimizer and schedule).
    Returns (avg_loss, avg_loss_components[3]) like the reference."""
    trainer.model.train()
    metrics = DeviceMetrics(trainer.device, log_every)
    n_batches = len(dataloader)
    step_fn = trainer.train_step_graphed if graphed else trainer.train_step
    for batch_idx, (image_tensor, labels_tensor) in enumerate(dataloader):
        if sequence_length is not None:
            image_tensor = image_tensor[:, :sequence_length]
        frames = image_tensor.to(trainer.device, non_blocking=True)
        batch = _batch_dict(trainer, labels_tensor, frames.shape[0], max_boxes)
        lr = trainer.lr()                                  # the rate this step runs at (host-side table lookup, no sync)
        _, items = step_fn(frames.contiguous(), batch)
        # the reference logs loss_components.sum() = B * sum(items) as 'Loss/train_batch' and the detached per-image
        # components (train.py:74-95); `items` are those detached components
        if metrics.update(items, epoch * n_batches + batch_idx, lr, scale=float(frames.shape[0])):
            _log_batches(writer, metrics.flush(), True)
    _log_batches(writer, metrics.flush(), True)
    return metrics.averages(n_batches)


@torch.no_grad()
def validate_one_epoch(trainer, dataloader, sequence_length=None, writer=None, epoch=0, log_every=50, max_boxes=None,
                       metrics=None, model=None):
    """reference train.py:106-146: eval mode, state reset per window, loss on the last frame.  `metrics`: a
    metrics.DetMetrics that also receives the detections of the same forwards (call its compute() afterwards).
    `model`: the network to validate (default trainer.model; trainer.ema.ema validates the weight average)."""
    det_metrics = metrics
    metrics = DeviceMetrics(trainer.device, log_every)
    n_batches = len(dataloader)
    for batch_idx, (image_tensor, labels_tensor) in enumerate(dataloader):
        if sequence_length is not None:
            image_tensor = image_tensor[:, :sequence_length]
        frames = image_tensor.to(trainer.device, non_blocking=True)
        batch = _batch_dict(trainer, labels_tensor, frames.shape[0], max_boxes)
        items = trainer.validate_step(frames.contiguous(), batch, metrics=det_metrics, model=model)
        if metrics.update(items, epoch * n_batches + batch_idx):
            _log_batches(writer, metrics.flush(), False)
    _log_batches(writer, metrics.flush(), False)
    return metrics.averages(n_batches)


def train_loop(model, train_loader, val_loader, config, device, save_dir, process_group=None, writer=None, log_every=50, graphed=False,
               max_boxes=None, eval_map=False, spike_stats=False, ema=False):
    """reference train.py:148-241: epochs of train + validation, `latest.pt` every epoch and `best.pt` on improvement (the
    reference's checkpoint dict, plus optimizer state), the reference's epoch-level TensorBoard tags.
    eval_map=True: the validation forwards also feed a DetMetrics, and metrics/{precision,recall,mAP50,mAP50-95}(B) are
    logged every epoch.
    spike_stats=True: one spikes.SpikeStats counts every forward of the loop; after each phase of an epoch it is read and
    reset, and Spikes/{train,val}_rate, Spikes/{train,val}_synops_fraction and the per-layer validation rates
    (Spikes_Val_Rate) are logged.  The model's previous `spike_stats` is restored on return.
    ema=True: an ema.ModelEMA (ultralytics' defaults) is updated after every optimizer step, and each epoch's validation --
    Loss/val and its components, metrics/*(B), the validation spike rates -- runs on the averaged weights, as ultralytics'
    trainer does; best.pt is chosen by that loss and both checkpoints carry the average under 'ema'.  The trainer's
    previous `ema` is restored on return.
    Returns the Trainer (the reference returns None)."""
    from .trainer import Trainer
    if writer is None:
        try:
            from torch.utils.tensorboard import SummaryWriter
            writer = SummaryWriter(log_dir=os.path.join(str(save_dir), "runs"))
        except Exception:
            writer = None
    tc = config["training"]
    total_steps = len(train_loader) * tc["epochs"]                          # train.py:161
    trainer = Trainer(model, max_lr=tc["learning_rate"], weight_decay=tc["weight_decay"], total_steps=max(1, total_steps),
                      device=device, process_group=process_group)
    seq_len = config["dataset"]["train"]["seq_len"]
    rank0 = (not torch.distributed.is_initialized()) or torch.distributed.get_rank() == 0
    det_metrics = None
    if eval_map:
        from .metrics import KEYS, DetMetrics
        det_metrics = DetMetrics(model.nc, trainer.device)
    prev_stats, stats = getattr(model, "spike_stats", None), None
    if spike_stats:
        from .spikes import MAX_T, SpikeStats
        stats = SpikeStats(model, max_T=MAX_T)       # one buffer for both phases: the training graph is captured once
        model.spike_stats = stats
    prev_ema, val_model = trainer.ema, model
    if ema:
        from .ema import ModelEMA
        trainer.ema = ModelEMA(model)
        val_model = trainer.ema.ema
        val_model.spike_stats = stats
    log = writer is not None and rank0
    best_val_loss = float("inf")
    try:
        for epoch in range(tc["epochs"]):
            sampler = getattr(train_loader, "sampler", None)
            if hasattr(sampler, "set_epoch"):
                sampler.set_epoch(epoch)
            train_loss, train_comps = train_one_epoch(trainer, train_loader, seq_len, writer=writer, epoch=epoch, log_every=log_every,
                                                      max_boxes=max_boxes, graphed=graphed)
            if stats is not None:
                res = _spike_results(stats, process_group)
                if log:
                    writer.add_scalar("Spikes/train_rate", res["spikes/rate"], epoch)
                    writer.add_scalar("Spikes/train_synops_fraction", res["spikes/synops_fraction"], epoch)
            if det_metrics is not None:
                det_metrics.reset()
            val_loss, val_comps = validate_one_epoch(trainer, val_loader, seq_len, writer=writer, epoch=epoch, log_every=log_every,
                                                     max_boxes=max_boxes, metrics=det_metrics, model=val_model)
            if stats is not None:
                res = _spike_results(stats, process_group)
                if log:
                    writer.add_scalar("Spikes/val_rate", res["spikes/rate"], epoch)
                    writer.add_scalar("Spikes/val_synops_fraction", res["spikes/synops_fraction"], epoch)
                    writer.add_scalars("Spikes_Val_Rate", {n: res["spikes/rate/" + n] for n in stats.layers}, epoch)
            if det_metrics is not None:
                res = det_metrics.compute(_metrics_group(process_group))
                if log:
                    for tag in KEYS[:4]:                        # metrics/{precision,recall,mAP50,mAP50-95}(B)
                        writer.add_scalar(tag, res[tag], epoch)
            if rank0:
                os.makedirs(str(save_dir), exist_ok=True)
                trainer.save_checkpoint(os.path.join(str(save_dir), "latest.pt"), epoch=epoch, best_val_loss=best_val_loss)
            if writer is not None and rank0:
                writer.add_scalar("Loss/train", train_loss, epoch)
                writer.add_scalar("Loss/val", val_loss, epoch)
                writer.add_scalar("LearningRate", trainer.lr(), epoch)
                writer.add_scalars("Train_Loss_Components", {k: float(v) for k, v in zip(COMPONENTS, train_comps)}, epoch)
                writer.add_scalars("Val_Loss_Components", {k: float(v) for k, v in zip(COMPONENTS, val_comps)}, epoch)
            if val_loss < best_val_loss:
                best_val_loss = val_loss
                if rank0:
                    trainer.save_checkpoint(os.path.join(str(save_dir), "best.pt"), epoch=epoch, best_val_loss=best_val_loss)
    finally:
        model.spike_stats = prev_stats
        if val_model is not model:
            val_model.spike_stats = None
        trainer.ema = prev_ema
    return trainer


def _spike_results(stats, process_group):
    """compute() + reset() of the loop's SpikeStats (all ranks take part in the all_reduce)."""
    res = stats.compute(_metrics_group(process_group))
    stats.reset()
    return res


def _metrics_group(process_group):
    """The group the detection records are gathered over: the trainer's, or the default one under torch.distributed."""
    if process_group is not None:
        return process_group
    if torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
        return torch.distributed.group.WORLD
    return None


@torch.no_grad()
def evaluate_model(model, dataloader, device, sequence_length=None, conf_thres=0.001, iou_thres=0.6, max_det=300,
                   process_group=None, spike_stats=False):
    """reference eval_2.py:20-130 as intended: every window of the loader through the eval-mode unroll (state reset per
    window), decode and NMS at eval_2.py:108's settings (conf 0.001, iou 0.6, best class per anchor), matched against the
    window's labels at IoU 0.50:0.05:0.95.  Returns DetMetrics.compute()'s dict: "metrics/precision(B)",
    "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)", "fitness", "ap", "ap_class_index".  Windows replay
    from one CUDA graph (GraphedWindowDetector); the host reads the device once, at the end.  Under data parallelism
    every rank evaluates its shard and gets the metric over all of them (see DetMetrics.compute).
    spike_stats=True: the windows are also counted by a spikes.SpikeStats, and the dict carries its "spikes/*" results
    (firing rates, SynOps, dense MACs) over the whole evaluation."""
    from .infer import GraphedWindowDetector
    from .loss import pad_targets
    from .metrics import DetMetrics
    device = torch.device(device)
    model.to(device)
    metrics = DetMetrics(model.nc, device)
    detector = GraphedWindowDetector(model, conf_thres=conf_thres, iou_thres=iou_thres, multi_label=False, max_det=max_det)
    prev_stats, stats = getattr(model, "spike_stats", None), None
    if spike_stats:
        from .spikes import MAX_T, SpikeStats
        stats = SpikeStats(model, max_T=MAX_T)
        model.spike_stats = stats
    try:
        for image_tensor, labels_tensor in dataloader:
            if sequence_length is not None:
                image_tensor = image_tensor[:, :sequence_length]
            frames = image_tensor.to(device, non_blocking=True).contiguous()
            rows, _, counts = detector(frames)
            metrics.update(rows, counts, pad_targets(labels_tensor, frames.shape[0]), frames.shape[-2:])
    finally:
        model.spike_stats = prev_stats
    res = metrics.compute(_metrics_group(process_group))
    if stats is not None:
        res.update((k, v) for k, v in stats.compute(_metrics_group(process_group)).items() if k.startswith("spikes/"))
    return res


# ------------------------------------------------------------------------------------------------
# input pipeline: sequence-grouped split (main.py:16-27) and the per-rank sampler over it
# ------------------------------------------------------------------------------------------------
def get_train_val_split(config, full_train_dataset, test_size=0.2, random_state=42):
    """reference main.py:16-27: whole recording sequences (grouped by image directory) go to train OR validation, 80/20,
    sklearn's train_test_split(random_state=42) so the split is the reference's.  Returns two torch Subsets."""
    from sklearn.model_selection import train_test_split
    from torch.utils.data import Subset
    seq_groups = defaultdict(list)
    for idx, (img_dir, _, _) in enumerate(full_train_dataset.samples):
        seq_groups[str(img_dir)].append(idx)
    train_seqs, val_seqs = train_test_split(list(seq_groups), test_size=test_size, random_state=random_state)
    train_seqs = set(train_seqs)
    train_indices, val_indices = [], []
    for seq, indices in seq_groups.items():
        (train_indices if seq in train_seqs else val_indices).extend(indices)
    return Subset(full_train_dataset, train_indices), Subset(full_train_dataset, val_indices)


class ShardedSampler(torch.utils.data.Sampler):
    """Per-rank sampler (DistributedSampler semantics) for one process per GPU: every epoch a permutation seeded by
    (seed, epoch) -- identical on all ranks -- is padded (or truncated with drop_last) to a multiple of world_size and
    rank r takes elements r, r+world, ...  With world_size 1 and shuffle=True it is DataLoader(shuffle=True) with a
    reproducible order (main.py:57-64).  The padding repeats samples: a distributed evaluation (evaluate_model,
    train_loop(eval_map=True)) counts the repeats like any other image, as with a stock DistributedSampler."""

    def __init__(self, data_source, rank=None, world_size=None, shuffle=True, seed=42, drop_last=False):
        if world_size is None:
            world_size = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
        if rank is None:
            rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        assert 0 <= rank < world_size
        self.n, self.rank, self.world, self.shuffle, self.seed, self.drop_last = len(data_source), rank, world_size, shuffle, seed, drop_last
        self.epoch = 0
        self.num_samples = self.n // world_size if drop_last else math.ceil(self.n / world_size)

    def set_epoch(self, epoch):
        self.epoch = int(epoch)

    def __len__(self):
        return self.num_samples

    def __iter__(self):
        if self.shuffle:
            g = torch.Generator().manual_seed(self.seed + self.epoch)
            order = torch.randperm(self.n, generator=g).tolist()
        else:
            order = list(range(self.n))
        total = self.num_samples * self.world
        if self.drop_last:
            order = order[:total]
        elif total > len(order) and order:
            order = (order * math.ceil(total / len(order)))[:total]
        return iter(order[self.rank:total:self.world])


def make_loaders(config, train_dataset, val_dataset, rank=None, world_size=None, seed=42):
    """DataLoaders of main.py:57-72 with a per-rank shard, pinned memory and the reference's collate layout."""
    from torch.utils.data import DataLoader
    tc = config["training"]
    tr_s = ShardedSampler(train_dataset, rank, world_size, shuffle=True, seed=seed)
    va_s = ShardedSampler(val_dataset, rank, world_size, shuffle=False, seed=seed)
    kw = dict(batch_size=tc["batch_size"], num_workers=tc.get("num_workers", 0), pin_memory=True, collate_fn=custom_collate_fn)
    return DataLoader(train_dataset, sampler=tr_s, **kw), DataLoader(val_dataset, sampler=va_s, **kw)
